// extern "C" surface of libopenpose_b200.so (include/openpose_b200.h) and the per-frame pipelines behind
// Body.__call__ (src/body.py:24-212) and Hand.__call__ (src/hand.py:25-75).
#include "net.cuh"
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <cmath>
#include <initializer_list>
#include <mutex>

namespace opb {

static thread_local std::string g_last_error;
void set_last_error(const std::string& m) { g_last_error = m; }

// OPB_DEBUG_ERRORS=1: report CUDA errors that are pending when an entry point is entered or left (an unchecked failing
// call of this library or of another CUDA user in the process would otherwise surface at some later launch check)
static void report_pending(const char* fn, const char* when) {
    static const bool on = getenv("OPB_DEBUG_ERRORS") != nullptr;
    if (!on) return;
    const cudaError_t e = cudaPeekAtLastError();
    if (e != cudaSuccess) fprintf(stderr, "[opb] pending CUDA error %s %s: %s\n", when, fn, cudaGetErrorString(e));
}

template <typename F>
static int guarded(F&& f, const char* fn = __builtin_FUNCTION()) {
    report_pending(fn, "on entry to");
    int rc = OPB_OK;
    try {
        f();
    } catch (const Error& e) {
        set_last_error(e.what());
        rc = e.code;
    } catch (const std::exception& e) {
        set_last_error(e.what());
        rc = OPB_ERR_INVALID;
    }
    report_pending(fn, "on return from");
    return rc;
}

struct ScaleDims {
    double mult;
    int h, w, hp, wp, ho, wo;
};
static ScaleDims scale_dims(int H, int W, double scale) {
    OPB_REQUIRE(H > 0 && W > 0, "empty image (the reference divides by oriImg.shape[0], src/body.py:32)");
    ScaleDims d;
    d.mult = scale * 368.0 / (double)H;                 // x * boxsize / oriImg.shape[0], src/body.py:32
    d.h = resize_dsize(H, d.mult);
    d.w = resize_dsize(W, d.mult);
    OPB_REQUIRE(d.h > 0 && d.w > 0, "scaled image is empty");
    d.hp = (d.h + 7) / 8 * 8;
    d.wp = (d.w + 7) / 8 * 8;
    d.ho = d.hp / 8;
    d.wo = d.wp / 8;
    return d;
}

// Tap tables of one frame plan are laid out in ONE host slab, copied with one stream-ordered transfer into one device
// allocation; the builders below return slab offsets disguised as pointers, relocated once the device base is known.
struct TableSlab {
    std::vector<uint8_t> host;
    template <typename T>
    T* add(const std::vector<T>& v) {
        const size_t off = (host.size() + 15) & ~(size_t)15;
        host.resize(off + std::max<size_t>(v.size(), 1) * sizeof(T));
        if (!v.empty()) memcpy(host.data() + off, v.data(), v.size() * sizeof(T));
        return (T*)off;
    }
};
template <typename T>
static void relocate(T*& p, uint8_t* base) { p = (T*)(base + (size_t)p); }
// device copy of a finished slab, ordered on `st` (the slab must outlive the copy)
static uint8_t* commit_tables(DevPool& pool, const TableSlab& slab, cudaStream_t st) {
    uint8_t* dev = (uint8_t*)pool.alloc(slab.host.size());
    OPB_CUDA(cudaMemcpyAsync(dev, slab.host.data(), slab.host.size(), cudaMemcpyHostToDevice, st));
    return dev;
}

// fixed-point (11-bit) tap tables of cv2's uint8 cubic resize
struct U8Taps {
    int *xf, *yf;
    short *xc, *yc;
    void relocate_to(uint8_t* b) { relocate(xf, b); relocate(yf, b); relocate(xc, b); relocate(yc, b); }
};
static std::vector<short> u8_coefs(const CubicTaps& t) {
    std::vector<short> out(t.coef.size());
    for (size_t i = 0; i < t.coef.size(); ++i) {
        long v = lrintf(t.coef[i] * 2048.0f);           // saturate_cast<short>(coef * INTER_RESIZE_COEF_SCALE)
        out[i] = (short)std::max(-32768l, std::min(32767l, v));
    }
    return out;
}
static U8Taps make_u8_taps(TableSlab& pool, int H, int W, const ScaleDims& d) {
    const CubicTaps tx = cubic_taps(W, d.w, 1.0 / d.mult), ty = cubic_taps(H, d.h, 1.0 / d.mult);
    U8Taps u;
    u.xf = pool.add(tx.first);
    u.yf = pool.add(ty.first);
    u.xc = pool.add(u8_coefs(tx));
    u.yc = pool.add(u8_coefs(ty));
    return u;
}
// cv2.resize(crop, (boxsize, boxsize), INTER_CUBIC) of a side x side crop (srcmx/Batch_model.py:96-101): dsize mode,
// inverse scale (double)boxsize / side, step = 1 / inverse scale
static CubicTaps hand_track_taps(int side, int boxsize) {
    return cubic_taps(side, boxsize, 1.0 / ((double)boxsize / side));
}

// Batch_body.calculate_size_pad (srcmx/Batch_model.py:340-345): truncating sizes, one scale; Batch_hand: no resize
static ScaleDims batch_dims(int H, int W, double g_scale, bool body) {
    OPB_REQUIRE(H > 0 && W > 0, "empty frame");
    ScaleDims d;
    if (body) {
        d.mult = 368.0 * g_scale / (double)H;
        d.h = (int)((double)H * d.mult);
        d.w = (int)((double)W * d.mult);
        OPB_REQUIRE(d.h > 0 && d.w > 0, "scaled frame is empty");
    } else {
        OPB_REQUIRE(H % 8 == 0 && W % 8 == 0, "Batch_hand crops must have sides that are multiples of 8 (the reference "
                                              "upsamples the stride-8 maps by exactly 8, srcmx/Batch_model.py:377)");
        d.mult = 1.0;
        d.h = H;
        d.w = W;
    }
    d.hp = (d.h + 7) / 8 * 8;
    d.wp = (d.w + 7) / 8 * 8;
    d.ho = d.hp / 8;
    d.wo = d.wp / 8;
    return d;
}

// float tap tables of the torch bicubic resize (batched estimators' front end)
struct F32Taps {
    int *xf, *yf;
    float *xc, *yc;
    void relocate_to(uint8_t* b) { relocate(xf, b); relocate(yf, b); relocate(xc, b); relocate(yc, b); }
};
static F32Taps make_f32_taps(TableSlab& pool, int H, int W, const ScaleDims& d) {
    const CubicTaps tx = cubic_taps(W, d.w, 1.0 / d.mult), ty = cubic_taps(H, d.h, 1.0 / d.mult);
    F32Taps u;
    u.xf = pool.add(tx.first);
    u.yf = pool.add(ty.first);
    u.xc = pool.add(tx.coef);
    u.yc = pool.add(ty.coef);
    return u;
}

struct UpTables {
    int *xf, *yf;
    float *xw, *yw;       // yw: 1/n_scales folded in
    int *ybf, *ybr;       // 8-row strip tables of the register-blocked y pass
    float* ybw;
    int yb_rs;
    // host copies / bounds for the fused peak kernel (peaks.cu)
    std::vector<int> h_xf, h_ybf, h_ybr;
    double l1 = 0, sum_min = 0, sum_max = 0;     // over all (y, x): sum |wy||wx| and range of (sum wy)(sum wx)
    void relocate_to(uint8_t* b) {
        relocate(xf, b); relocate(yf, b); relocate(xw, b); relocate(yw, b);
        relocate(ybf, b); relocate(ybr, b); relocate(ybw, b);
    }
};
static UpTables make_up_tables(TableSlab& pool, int H, int W, const ScaleDims& d, int n_scales) {
    std::vector<int> fx, fy;
    std::vector<float> wx, wy;
    composite_taps(d.wo, d.w, W, fx, wx);
    composite_taps(d.ho, d.h, H, fy, wy);
    // the cross-scale average (heatmap / len(multiplier), src/body.py:67-68) is folded into the row weights
    for (auto& v : wy) v = v / (float)n_scales;
    UpTables t;
    t.xf = pool.add(fx);
    t.yf = pool.add(fy);
    t.xw = pool.add(wx);
    t.yw = pool.add(wy);
    // strips of 8 output rows: first source row, number of source rows, dense weights
    const int TY = kUpStrip, nyb = (H + TY - 1) / TY;
    std::vector<int> bf(nyb), br(nyb);
    int rs = 1;
    for (int b = 0; b < nyb; ++b) {
        int lo = d.ho, hi = -1;
        for (int y = b * TY; y < std::min(H, (b + 1) * TY); ++y) {
            lo = std::min(lo, fy[y]);
            hi = std::max(hi, std::min(fy[y] + kUpTaps - 1, d.ho - 1));
        }
        bf[b] = lo;
        br[b] = hi - lo + 1;
        rs = std::max(rs, br[b]);
    }
    std::vector<float> bw((size_t)nyb * rs * TY, 0.f);
    for (int b = 0; b < nyb; ++b)
        for (int y = b * TY; y < std::min(H, (b + 1) * TY); ++y)
            for (int k = 0; k < kUpTaps; ++k) {
                const int r = std::min(fy[y] + k, d.ho - 1) - bf[b];      // same clamp as the generic kernel
                bw[((size_t)b * rs + r) * TY + (y - b * TY)] += wy[(size_t)y * kUpTaps + k];
            }
    t.ybf = pool.add(bf);
    t.ybr = pool.add(br);
    t.ybw = pool.add(bw);
    t.yb_rs = rs;
    auto axis = [](const std::vector<float>& w, double& l1, double& smin, double& smax) {
        l1 = 0; smin = 1e300; smax = -1e300;
        for (size_t i = 0; i < w.size(); i += kUpTaps) {
            double a = 0, sgn = 0;
            for (int k = 0; k < kUpTaps; ++k) { a += std::fabs((double)w[i + k]); sgn += (double)w[i + k]; }
            l1 = std::max(l1, a); smin = std::min(smin, sgn); smax = std::max(smax, sgn);
        }
    };
    double l1x, l1y, sxl, sxh, syl, syh;
    axis(wx, l1x, sxl, sxh);
    axis(wy, l1y, syl, syh);
    t.l1 = l1x * l1y;
    const double c[4] = {sxl * syl, sxl * syh, sxh * syl, sxh * syh};
    t.sum_min = *std::min_element(c, c + 4);
    t.sum_max = *std::max_element(c, c + 4);
    t.h_xf = fx;
    t.h_ybf = bf;
    t.h_ybr = br;
    return t;
}

// ------------------------------------------------------------------------------------------------
// frame plans
// ------------------------------------------------------------------------------------------------
struct FrameKey {
    int n, H, W;
    std::vector<double> scales;
    int mode = 0;               // 0: Body / Hand (src/); Batch_body / Batch_hand (srcmx/Batch_model.py): 1 float planar
                                // frames, 2 decoded uint8 HWC frames (ToTensor's /255 on the device)
    bool operator<(const FrameKey& o) const {
        if (mode != o.mode) return mode < o.mode;
        if (n != o.n) return n < o.n;
        if (H != o.H) return H < o.H;
        if (W != o.W) return W < o.W;
        return scales < o.scales;
    }
};

struct FramePlan {
    DevPool pool;
    FrameKey key;
    // the device work of one submit (everything between the input upload and the "done" event) as a CUDA graph:
    // captured on the third use of the plan, re-captured when a session buffer it points into has moved
    cudaGraphExec_t graph = nullptr;
    uint64_t graph_gen = 0;
    int uses = 0;
    // the same for the body + hands sequence of opb_pose_submit_batch (a different launch list over the same buffers)
    cudaGraphExec_t pose_graph = nullptr;
    uint64_t pose_gen = 0;
    int pose_uses = 0;
    // the same for the hand-track sequence of opb_hand_track_submit (a uint8 Batch_hand plan fed by the crop kernel)
    cudaGraphExec_t track_graph = nullptr;
    uint64_t track_gen = 0;
    int track_uses = 0;
    // the same for the one-pass body + hand sequence of opb_batch_pose_submit (on the Batch_body plan)
    cudaGraphExec_t batch_pose_graph = nullptr;
    uint64_t batch_pose_gen = 0;
    int batch_pose_uses = 0;
    // every person (opb_pose_every_*): the body sequence with the rows-and-boxes kernel, and one hand chunk (replayed
    // once per kEveryChunk boxes) -- both on the body plan of the batch.  opb_batch_pose_every_submit uses the same two
    // slots of its Batch_body plan (a mode-2 plan, which no other every-person sequence shares), so it alternates with
    // opb_batch_pose_submit (batch_pose_graph) on one session pair without re-capturing.
    cudaGraphExec_t every_graph = nullptr;
    uint64_t every_gen = 0;
    int every_uses = 0;
    cudaGraphExec_t every_hand_graph = nullptr;
    uint64_t every_hand_gen = 0;
    int every_hand_uses = 0;
    // Hand()(list of square crops) (opb_hand_submit_ragged), on the hand plan of the list
    cudaGraphExec_t crops_graph = nullptr;
    uint64_t crops_gen = 0;
    int crops_uses = 0;
    ~FramePlan() {
        if (crops_graph) cudaGraphExecDestroy(crops_graph);
        if (graph) cudaGraphExecDestroy(graph);
        if (pose_graph) cudaGraphExecDestroy(pose_graph);
        if (track_graph) cudaGraphExecDestroy(track_graph);
        if (batch_pose_graph) cudaGraphExecDestroy(batch_pose_graph);
        if (every_graph) cudaGraphExecDestroy(every_graph);
        if (every_hand_graph) cudaGraphExecDestroy(every_hand_graph);
    }
    std::vector<ScaleDims> dims;
    std::vector<U8Taps> u8taps;
    std::vector<F32Taps> f32taps;
    std::vector<UpTables> uptabs;
    NetPlan* net = nullptr;         // owned by the session's cache: shared by every frame size with the same net input
    TableSlab tables;               // host copy stays alive until the plan dies (source of an asynchronous copy)
    bool fused_ok = false;          // tile footprints of the heat maps fit the fused peak kernel
    // bound from the session's arenas at every submit (one plan is in flight per session)
    uint8_t* d_img = nullptr;
    // materialised full-resolution maps: hand crops always; body frames only when a caller asks for them
    // (opb_body_maps / opb_batch_maps) or when the fused peak kernel does not fit the resize ratio
    float* up_scratch = nullptr;
    float* heat_avg = nullptr;      // body: (n*19,H,W); hand: (n*22,H,W)
    float* paf_avg = nullptr;       // body: (n*38,H,W)
    float* blurred = nullptr;       // batched estimators: 5x5-blurred heat maps, same shape as heat_avg
    size_t scratch_floats = 0;
    // body post-processing: one FramePost per frame of the batch, a device copy of the table, one counter slab and
    // one result slab for the whole batch
    std::vector<FramePost> post;
    FramePost* post_dev = nullptr;
    int* counters = nullptr;        // [n][kCounterInts], cleared once per batch
    unsigned* tile_mask = nullptr;  // [n][tiles] parts that can hold a peak, per tile of the peak kernel
    FrameResults* results_dev = nullptr;
    // hand post-processing
    HandBuffers hb{};
    int launches_per_frame = 0;
};

constexpr int kCounterInts = 128;
constexpr int kPeakCapacity = 16384;
constexpr int kPairCapacity = 16384;
constexpr int kConnCapacity = 2048;
constexpr int kSubsetCapacity = kSubsetRowsShared;

// counters: [0] peaks appended, [1] ordering ticket, [2..19] part counts, [20..38] part_begin, [40..58] survivors per
// limb, [60..63] status, [64] subset rows, [65..83] connections per limb
static void alloc_body_post(DevPool& pool, FramePost& fp, int* counters, FrameResults* result, int peak_cap, int pair_cap,
                            int conn_cap, int subset_cap) {
    fp.pb.capacity = peak_cap;
    fp.pb.keys = pool.alloc_t<unsigned long long>(peak_cap);
    fp.pb.scores = pool.alloc_t<float>(peak_cap);
    fp.pb.count = counters + 0;
    fp.pb.ticket = counters + 1;
    fp.pb.part_count = counters + 2;
    fp.pb.part_begin = counters + 20;
    fp.pb.candidates = pool.alloc_t<double>((size_t)peak_cap * 4, true);
    fp.lb.pair_capacity = pair_cap;
    fp.lb.conn_capacity = conn_cap;
    fp.lb.subset_capacity = subset_cap;
    fp.lb.max_part = peak_cap;
    fp.lb.cand_score = pool.alloc_t<double>((size_t)19 * pair_cap);
    fp.lb.cand_ij = pool.alloc_t<int>((size_t)19 * pair_cap * 2);
    fp.lb.cand_count = counters + 40;
    fp.lb.status = counters + 60;
    fp.lb.subset_count = counters + 64;
    fp.lb.conn_count = counters + 65;
    fp.lb.conn = pool.alloc_t<double>((size_t)19 * conn_cap * 5, true);
    fp.lb.subset = pool.alloc_t<double>((size_t)subset_cap * 20, true);
    fp.lb.rows_global = subset_cap > kSubsetRowsShared ? pool.alloc_t<double>((size_t)subset_cap * kSubsetRowStride) : nullptr;
    fp.lb.order = pool.alloc_t<int>((size_t)19 * pair_cap);
    fp.lb.owner_global = pool.alloc_t<int4>((size_t)peak_cap);
    fp.lb.claim_global = subset_cap > kSubsetRowsShared ? pool.alloc_t<int>((size_t)subset_cap) : nullptr;
    fp.result = result;
}

}  // namespace opb

using namespace opb;

typedef FrameResults HostResults;    // pinned, one per frame of a body batch (same layout as the device block)
struct FrameResult {                 // host-side view of one finished frame
    int n_cand = 0, n_subset = 0, status = 0;
    std::vector<double> cand_all, subset_all;   // filled by wait() when the eager copy was too small
};

struct opb_session {
    opb_net* net = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    std::map<FrameKey, std::unique_ptr<FramePlan>> plans;
    FramePlan* active = nullptr;
    HostResults* host = nullptr;     // pinned, [frames]
    double* hand_host = nullptr;     // pinned, [crops][21][3]
    size_t host_bytes = 0, hand_host_bytes = 0;
    std::vector<FrameResult> results;
    int n_frames = 0;
    uint8_t* staging = nullptr;      // pinned image staging
    size_t staging_bytes = 0;
    int hand_crops = 0;
    Profiler prof;
    cudaEvent_t marks[2] = {nullptr, nullptr};
    // CNN plans keyed by the net input shapes only: every frame / crop size that resizes to the same shapes (all
    // square hand crops do: 184..736 squared, src/hand.py:38) shares one set of activations and tensor maps
    struct NetEntry {
        std::unique_ptr<NetPlan> plan;
        uint64_t last_use = 0;
    };
    std::map<std::vector<NetShape>, NetEntry> net_plans;
    uint64_t use_clock = 0;
    // size-dependent work buffers, grown to the largest frame seen and shared by all plans of the session
    enum { AR_IMG, AR_SCRATCH, AR_HEAT, AR_PAF, AR_LABELS, AR_SUMS, AR_PEAKS, AR_BLUR, AR_COUNT };
    struct Arena { void* p = nullptr; size_t cap = 0; } arena[AR_COUNT];
    uint64_t buffer_gen = 1;         // bumped whenever an arena or a pinned result buffer is reallocated
    // per-frame caller on the device (opb_pose_*): a hand session carries the tap tables of every crop size, a body
    // session the per-batch pose / box buffers
    struct Ragged {
        DevPool pool;
        std::vector<double> scales;
        RaggedTables tabs{};
        std::vector<int> net_side;   // net input side per scale (the same for every crop size)
    };
    std::unique_ptr<Ragged> ragged;
    // Hand()(list of square crops of any sides) (opb_hand_submit_ragged), on a hand session: the same tables for sides
    // up to the largest seen, kept apart from `ragged` (a pose batch of another stream may be reading those), and the
    // per-crop boxes, sides and byte offsets into the packed crops, grown to the longest list seen
    std::unique_ptr<Ragged> crop_tables;
    struct CropList {
        DevPool pool;
        int cap = 0;
        HandBox* boxes = nullptr;        // [cap] (x = y = 0, side, not mirrored)
        int* sides = nullptr;            // [cap]
        size_t* offsets = nullptr;       // [cap] byte offset of each crop in the packed input
        HandBox* boxes_host = nullptr;   // pinned copies, uploaded inside the launch sequence
        int* sides_host = nullptr;
        size_t* offsets_host = nullptr;
        ~CropList() {
            if (boxes_host) cudaFreeHost(boxes_host);
            if (sides_host) cudaFreeHost(sides_host);
            if (offsets_host) cudaFreeHost(offsets_host);
        }
    };
    std::unique_ptr<CropList> crop_list;
    bool hand_ragged = false;            // the last hand batch was a crop list: its maps have one pitch per crop
    struct PoseBuffers {
        DevPool pool;
        int frames = 0;
        double* pose = nullptr;      // [frames][60][3]
        HandBox* boxes = nullptr;    // [frames][2]
        int* dims = nullptr;         // [frames][2]
        int* fixed = nullptr;        // [frames][2][3]
        double* host = nullptr;      // pinned [frames][60][3]
        int* fixed_host = nullptr;   // pinned
        ~PoseBuffers() {
            if (host) cudaFreeHost(host);
            if (fixed_host) cudaFreeHost(fixed_host);
        }
    };
    std::unique_ptr<PoseBuffers> pose;
    // the batched hand job on saved poses (opb_hand_track_*), on a hand session: tap tables of every crop side for one
    // boxsize, and per-batch buffers grown to the largest batch / frame seen
    struct HandTrack {
        DevPool table_pool;
        RaggedTables tabs{};         // one "scale": crop side -> boxsize, preprocess entries only
        int boxsize = 0;
        DevPool pool, frame_pool;
        int frames = 0;              // capacity of the per-frame buffers
        size_t frame_bytes = 0;      // capacity of `frames_dev`
        uint8_t* frames_dev = nullptr;   // the decoded (ROI-cropped) frames of the batch
        double* poses = nullptr;     // [frames][18][3]
        HandBox* boxes = nullptr;    // [frames][2]
        double* mats = nullptr;      // [frames][42][3]
        double* poses_host = nullptr;   // pinned
        double* mats_host = nullptr;    // pinned
        uint64_t gen = 1;            // bumped whenever a buffer, the tables or the frame size change
        int H = 0, W = 0, n = 0;     // last batch
        FramePlan* plan = nullptr;   // uint8 Batch_hand plan of the last batch (its input buffer holds the crops)
        ~HandTrack() {
            if (poses_host) cudaFreeHost(poses_host);
            if (mats_host) cudaFreeHost(mats_host);
        }
    };
    std::unique_ptr<HandTrack> track;
    opb_session* pose_hand = nullptr;    // hand session of the pose batch in flight
    std::vector<double> pose_hand_scales;
    bool pose_fixed = false;
    int batch_pose_box = 0;              // boxsize of the opb_batch_pose(_every) batch in flight; 0: an opb_pose batch
    // every person of a batch (opb_pose_every_*), on a body session: the records and the compacted hand boxes, grown to
    // the largest person count seen, and the boxes of one hand chunk
    struct EveryBuffers {
        DevPool pool;
        int cap = 0;                 // records; the box list holds 2 * cap
        uint64_t gen = 0;            // unique per allocation (graph keys)
        double* records = nullptr;   // [cap][60][3]
        HandBox* list = nullptr;     // [2 cap] in util.handDetect's order
        int* list_rec = nullptr;     // [2 cap] record of each box
        int* counts = nullptr;       // [kEveryCounts] persons, boxes, chunk cursor
        HandBox* chunk_boxes = nullptr;  // [kEveryChunkSlots]
        int* chunk_dims = nullptr;       // [kEveryChunkSlots]
        int* chunk_rec = nullptr;        // [kEveryChunkSlots]
        double* records_host = nullptr;  // pinned [cap][60][3]
        int* counts_host = nullptr;      // pinned [kEveryCounts]
        int* ids = nullptr;              // [cap] track id of each record (opb_pose_every_wait_tracked)
        int* ids_host = nullptr;         // pinned [cap]
        ~EveryBuffers() {
            if (records_host) cudaFreeHost(records_host);
            if (counts_host) cudaFreeHost(counts_host);
            if (ids_host) cudaFreeHost(ids_host);
        }
    };
    std::unique_ptr<EveryBuffers> every;
    uint64_t every_allocs = 0;
    bool every_batch = false;            // the batch in flight is an opb_pose_every or opb_batch_pose_every batch
    int every_persons = -1;              // persons of the last finished opb_pose_every batch; -1: none
    bool every_linked = false;           // the last finished opb_pose_every batch was linked: ids_host holds its ids
    std::vector<NetShape> debug_shapes;  // the plan of the opb_net_debug_* calls (looked up by its shapes on every call)
    ~opb_session() {
        plans.clear();
        net_plans.clear();
        for (auto& a : arena) if (a.p) cudaFree(a.p);
        if (host) cudaFreeHost(host);
        if (hand_host) cudaFreeHost(hand_host);
        if (staging) cudaFreeHost(staging);
        if (done) cudaEventDestroy(done);
        for (auto m : marks) if (m) cudaEventDestroy(m);
        if (stream) cudaStreamDestroy(stream);
    }
};

// person tracks of one video (track.cu).  The host holds the authoritative (cur, live, next_id, frame); every link
// passes it to the kernel and reads it back before it returns, under `mu`.
struct opb_tracker {
    opb_context* ctx = nullptr;
    int max_gap = 1, min_joints = 3;
    double max_dist = 0.0;
    std::mutex mu;
    int cur = 0, live = 0, next_id = 0, frame = 0;
    // track slots (double-buffered), grown by doubling with the live tracks carried over
    opb::DevPool tracks;
    int cap = 0;
    double* rows[2] = {nullptr, nullptr};
    int* tid[2] = {nullptr, nullptr};
    int* last[2] = {nullptr, nullptr};
    int* track_taken = nullptr;
    // per-frame scratch
    opb::DevPool scratch;
    int person_cap = 0, pair_cap = 0;
    int* match = nullptr;
    double* pair_cost = nullptr;
    int* pair_k = nullptr;
    int* pair_p = nullptr;
    int* order = nullptr;
    int* state = nullptr;             // [5] kernel output
    int* state_host = nullptr;        // pinned [5]
    // opb_tracker_link_host: the caller's records in device memory
    opb::DevPool staging;
    int staging_records = -1, staging_frames = -1;
    double* records = nullptr;
    int* persons = nullptr;
    int* ids = nullptr;
    ~opb_tracker() {
        if (state_host) cudaFreeHost(state_host);
    }
};

namespace opb {

static void ensure_host(opb_session* s, int frames, size_t hand_doubles) {
    const size_t need = sizeof(HostResults) * (size_t)frames;
    if (s->host_bytes < need) {
        if (s->host) cudaFreeHost(s->host);
        OPB_CUDA(cudaMallocHost((void**)&s->host, need));
        s->host_bytes = need;
        ++s->buffer_gen;
    }
    const size_t hneed = hand_doubles * sizeof(double);
    if (s->hand_host_bytes < hneed) {
        if (s->hand_host) cudaFreeHost(s->hand_host);
        OPB_CUDA(cudaMallocHost((void**)&s->hand_host, hneed));
        s->hand_host_bytes = hneed;
        ++s->buffer_gen;
    }
}
static void ensure_staging(opb_session* s, size_t bytes) {
    if (s->staging_bytes >= bytes) return;
    if (s->staging) cudaFreeHost(s->staging);
    OPB_CUDA(cudaMallocHost((void**)&s->staging, bytes));
    s->staging_bytes = bytes;
}

constexpr size_t kMaxFramePlans = 512;     // tap tables only (tens of KB each)
constexpr size_t kMaxNetPlans = 6;         // activations + tensor maps (hundreds of MB each)

static void drop_plans(opb_session* s) {
    OPB_CUDA(cudaStreamSynchronize(s->stream));
    s->plans.clear();
    s->active = nullptr;
}

// Plan construction allocates with cudaMalloc, uploads with synchronous copies and zero-fills through DevPool (which
// waits for its own fill): nothing of it is ordered against, or waits for, the other sessions' streams.  When the
// cache is full the least recently used CNN plan goes, together with the frame plans that point at it.
static NetPlan* get_net_plan(opb_session* s, const std::vector<NetShape>& shapes) {
    auto it = s->net_plans.find(shapes);
    if (it != s->net_plans.end()) {
        it->second.last_use = ++s->use_clock;
        return it->second.plan.get();
    }
    if (s->net_plans.size() >= kMaxNetPlans) {
        auto victim = s->net_plans.begin();
        for (auto jt = s->net_plans.begin(); jt != s->net_plans.end(); ++jt)
            if (jt->second.last_use < victim->second.last_use) victim = jt;
        OPB_CUDA(cudaStreamSynchronize(s->stream));             // this session's work only
        const NetPlan* dead = victim->second.plan.get();
        for (auto pt = s->plans.begin(); pt != s->plans.end();) {
            if (pt->second->net == dead) {
                if (s->active == pt->second.get()) s->active = nullptr;
                pt = s->plans.erase(pt);
            } else {
                ++pt;
            }
        }
        s->net_plans.erase(victim);
    }
    auto plan = build_net_plan(s->net, shapes);
    NetPlan* raw = plan.get();
    auto& e = s->net_plans[shapes];
    e.plan = std::move(plan);
    e.last_use = ++s->use_clock;
    return raw;
}

static void* arena_get(opb_session* s, int which, size_t bytes) {
    auto& a = s->arena[which];
    if (a.cap < bytes) {
        OPB_CUDA(cudaStreamSynchronize(s->stream));
        if (a.p) OPB_CUDA(cudaFree(a.p));
        a.p = nullptr;
        a.cap = 0;
        const size_t want = bytes + bytes / 4 + 256;
        OPB_CUDA(cudaMalloc(&a.p, want));
        a.cap = want;
        ++s->buffer_gen;
    }
    return a.p;
}

// points the plan's work buffers at the session's arenas (which may have grown or moved since the last use)
static void bind_maps(opb_session* s, FramePlan* fp, bool heat, bool paf, bool blurred) {
    const size_t n = fp->key.n, px = (size_t)fp->key.H * fp->key.W;
    const bool body = s->net->kind == OPB_NET_BODY;
    fp->up_scratch = (float*)arena_get(s, opb_session::AR_SCRATCH, fp->scratch_floats * sizeof(float));
    if (heat) fp->heat_avg = (float*)arena_get(s, opb_session::AR_HEAT, n * (body ? 19 : 22) * px * sizeof(float));
    if (paf) fp->paf_avg = (float*)arena_get(s, opb_session::AR_PAF, n * 38 * px * sizeof(float));
    if (blurred) fp->blurred = (float*)arena_get(s, opb_session::AR_BLUR, n * (body ? 19 : 22) * px * sizeof(float));
}

static void bind_buffers(opb_session* s, FramePlan* fp) {
    const size_t n = fp->key.n, px = (size_t)fp->key.H * fp->key.W;
    const bool body = s->net->kind == OPB_NET_BODY;
    const bool batch_mode = fp->key.mode >= 1;
    fp->d_img = (uint8_t*)arena_get(s, opb_session::AR_IMG, n * px * 3 * (fp->key.mode == 1 ? sizeof(float) : 1));
    if (body) {
        // the full-resolution maps are not materialised (peaks.cu / paf.cu evaluate them on the fly) unless the
        // resize ratio is outside what the fused kernel's shared memory holds
        if (!fp->fused_ok) bind_maps(s, fp, true, false, false);
    } else {
        bind_maps(s, fp, true, false, batch_mode);
        fp->hb.labels = (int*)arena_get(s, opb_session::AR_LABELS, n * 21 * px * sizeof(int));
        fp->hb.sums = (double*)arena_get(s, opb_session::AR_SUMS, n * 21 * px * sizeof(double));
        fp->hb.peaks = (double*)arena_get(s, opb_session::AR_PEAKS, n * 21 * 3 * sizeof(double));
    }
}

static void upload_post_table(FramePlan* fp, cudaStream_t st) {
    OPB_CUDA(cudaMemcpyAsync(fp->post_dev, fp->post.data(), fp->post.size() * sizeof(FramePost), cudaMemcpyHostToDevice, st));
}

// per-scale net output sizes of a plan: mode 0 Body (scale_search), mode >= 1 the batched estimators (one scale)
static ScaleDims plan_dims(int H, int W, double scale, int mode, bool body) {
    return mode >= 1 ? batch_dims(H, W, scale, body) : scale_dims(H, W, scale);
}

// do the heat maps of a body plan fit the fused peak kernel (peaks.cu), so that they need not be materialised?
static bool plan_fits_fused(const std::vector<UpTables>& uptabs, const std::vector<ScaleDims>& dims, int H, int W) {
    std::vector<std::vector<int>> xf, ybf, ybr;
    std::vector<int> wo, rs;
    for (size_t i = 0; i < dims.size(); ++i) {
        xf.push_back(uptabs[i].h_xf);
        ybf.push_back(uptabs[i].h_ybf);
        ybr.push_back(uptabs[i].h_ybr);
        wo.push_back(dims[i].wo);
        rs.push_back(uptabs[i].yb_rs);
    }
    return composite_fits_fused(xf, ybf, ybr, wo, rs, H, W);
}

static FramePlan* get_plan(opb_session* s, int n, int H, int W, const double* scales, int n_scales, int mode = 0) {
    OPB_REQUIRE(n_scales >= 1 && n_scales <= kMaxScales, "scale_search must hold 1..8 entries");
    FrameKey key{n, H, W, std::vector<double>(scales, scales + n_scales), mode};
    auto it = s->plans.find(key);
    if (it != s->plans.end()) {
        FramePlan* fp = it->second.get();
        auto nt = s->net_plans.find(fp->net->shapes);
        if (nt != s->net_plans.end()) nt->second.last_use = ++s->use_clock;
        bind_buffers(s, fp);
        return fp;
    }
    OPB_CUDA(cudaSetDevice(s->net->ctx->device));
    if (s->plans.size() >= kMaxFramePlans) drop_plans(s);
    auto fp = std::make_unique<FramePlan>();
    fp->key = key;
    const bool body = s->net->kind == OPB_NET_BODY;
    std::vector<NetShape> shapes;
    const int C = body ? 57 : 22;
    for (int i = 0; i < n_scales; ++i) {
        const ScaleDims d = plan_dims(H, W, scales[i], mode, body);
        fp->dims.push_back(d);
        if (mode >= 1) fp->f32taps.push_back(make_f32_taps(fp->tables, H, W, d));
        else fp->u8taps.push_back(make_u8_taps(fp->tables, H, W, d));
        fp->uptabs.push_back(make_up_tables(fp->tables, H, W, d, n_scales));
        shapes.push_back({n, d.hp, d.wp, mode >= 1 ? 2 : 1});
        fp->scratch_floats += (size_t)n * C * d.ho * W;
    }
    fp->net = get_net_plan(s, shapes);          // may evict another CNN plan of the session (and its frame plans)
    // tables: one device allocation, one copy ordered on the session's stream (no device-wide synchronisation, so a
    // new crop size on one session does not stall the others)
    uint8_t* dev_tables = commit_tables(fp->pool, fp->tables, s->stream);
    for (auto& t : fp->u8taps) t.relocate_to(dev_tables);
    for (auto& t : fp->f32taps) t.relocate_to(dev_tables);
    for (auto& t : fp->uptabs) t.relocate_to(dev_tables);
    fp->launches_per_frame = n_scales /*preprocess*/ + fp->net->kernel_launches;
    if (body) {
        static const bool no_fuse = getenv("OPB_NO_FUSED_PEAKS") != nullptr;      // A/B switch: materialised planes
        fp->fused_ok = !no_fuse && plan_fits_fused(fp->uptabs, fp->dims, H, W);
        // OPB_TEST_SMALL_BUFFERS: start with tiny result buffers so that tests exercise the growth path of body_wait
        static const bool tiny = getenv("OPB_TEST_SMALL_BUFFERS") != nullptr;
        fp->counters = fp->pool.alloc_t<int>((size_t)n * kCounterInts, true);
        fp->results_dev = fp->pool.alloc_t<FrameResults>(n, true);
        fp->post_dev = fp->pool.alloc_t<FramePost>(n);
        fp->tile_mask = fp->pool.alloc_t<unsigned>(find_peaks_mask_words(n, H, W));
        fp->post.resize(n);
        for (int f = 0; f < n; ++f)
            alloc_body_post(fp->pool, fp->post[f], fp->counters + (size_t)f * kCounterInts, fp->results_dev + f,
                            tiny ? 64 : kPeakCapacity, tiny ? 64 : kPairCapacity, tiny ? 16 : kConnCapacity,
                            tiny ? 4 : kSubsetCapacity);
        upload_post_table(fp.get(), s->stream);
        fp->launches_per_frame += 8 + (fp->fused_ok ? 0 : n_scales + 1);   // bounds, peaks, order, score, sort, match, assemble, pack
    } else {
        fp->launches_per_frame += (n_scales + 1) + 6 + (mode >= 1);
    }
    bind_buffers(s, fp.get());
    FramePlan* raw = fp.get();
    s->plans[key] = std::move(fp);
    return raw;
}

// Runs `enqueue` (kernel launches, memsets and result copies on the session's stream) either directly or, once the plan
// has been used a few times, as one CUDA graph launch: a frame is ~70 small dependent launches, and for the small
// default configuration (640x480, one scale) the launch gaps, not the kernels, are most of the latency.
struct GraphSlot {
    cudaGraphExec_t& graph;
    uint64_t& gen;
    int& uses;
};
template <typename F>
static void run_or_replay_slot(opb_session* s, GraphSlot g, uint64_t want_gen, F&& enqueue) {
    static const bool no_graph = getenv("OPB_NO_GRAPH") != nullptr;
    cudaStream_t st = s->stream;
    ++g.uses;
    if (no_graph || s->prof.on || g.uses < 3) {         // first uses run eagerly (lazy module loading, attributes)
        enqueue();
        return;
    }
    if (!g.graph || g.gen != want_gen) {
        if (g.graph) {
            cudaGraphExecDestroy(g.graph);
            g.graph = nullptr;
        }
        cudaGraph_t cg = nullptr;
        OPB_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
        try {
            enqueue();
        } catch (...) {
            cudaStreamEndCapture(st, &cg);
            if (cg) cudaGraphDestroy(cg);
            throw;
        }
        OPB_CUDA(cudaStreamEndCapture(st, &cg));
        const cudaError_t e = cudaGraphInstantiate(&g.graph, cg, 0);
        cudaGraphDestroy(cg);
        OPB_CUDA(e);
        g.gen = want_gen;
    }
    OPB_CUDA(cudaGraphLaunch(g.graph, st));
}
template <typename F>
static void run_or_replay(opb_session* s, FramePlan* fp, F&& enqueue) {
    run_or_replay_slot(s, GraphSlot{fp->graph, fp->graph_gen, fp->uses}, s->buffer_gen, enqueue);
}

static void upload_bytes(opb_session* s, void* dst, const void* img, int where, size_t bytes) {
    if (where == 1) {                                    // already on the device
        OPB_CUDA(cudaMemcpyAsync(dst, img, bytes, cudaMemcpyDeviceToDevice, s->stream));
    } else if (where == 2) {                             // caller-owned pinned host memory
        OPB_CUDA(cudaMemcpyAsync(dst, img, bytes, cudaMemcpyHostToDevice, s->stream));
    } else {                                             // pageable host memory: stage through pinned
        ensure_staging(s, bytes);
        OPB_CUDA(cudaStreamSynchronize(s->stream));      // staging buffer may still feed the previous frame
        memcpy(s->staging, img, bytes);
        OPB_CUDA(cudaMemcpyAsync(dst, s->staging, bytes, cudaMemcpyHostToDevice, s->stream));
    }
}
static void upload_image(opb_session* s, FramePlan* fp, const uint8_t* img, int where, size_t bytes) {
    upload_bytes(s, fp->d_img, img, where, bytes);
}

static void run_front(opb_session* s, FramePlan* fp, int n, int H, int W) {
    cudaStream_t st = s->stream;
    const int S = (int)fp->dims.size();
    for (int i = 0; i < S; ++i) {
        const ScaleDims& d = fp->dims[i];
        const U8Taps& t = fp->u8taps[i];
        preprocess_launch_batched(fp->d_img, n, H, W, fp->net->in_u8[i], d.h, d.w, d.hp, d.wp, t.xf, t.xc, t.yf, t.yc, st);
    }
    s->prof.mark(st, "preprocess");
    fp->net->run(st, s->prof.on ? &s->prof : nullptr);
}

// materialises the averaged full-resolution maps (hand crops; body maps on request)
static void run_upsample(FramePlan* fp, bool paf, int n, int C, int cstride, int H, int W, float* out, cudaStream_t st) {
    UpsampleScale us[kMaxScales];
    const int S = (int)fp->dims.size();
    for (int i = 0; i < S; ++i) {
        us[i].src = paf ? fp->net->out_paf[i] : fp->net->out_heat[i];
        us[i].ho = fp->dims[i].ho;
        us[i].wo = fp->dims[i].wo;
        us[i].cstride = cstride;
        us[i].x_first = fp->uptabs[i].xf;
        us[i].x_w = fp->uptabs[i].xw;
        us[i].y_first = fp->uptabs[i].yf;
        us[i].y_w = fp->uptabs[i].yw;
        us[i].yb_first = fp->uptabs[i].ybf;
        us[i].yb_rows = fp->uptabs[i].ybr;
        us[i].yb_w = fp->uptabs[i].ybw;
        us[i].yb_rs = fp->uptabs[i].yb_rs;
    }
    upsample_avg_launch2(us, S, n, C, H, W, fp->up_scratch, out, st);
}

// the averaged map as a function of the net outputs (peaks.cu, paf.cu evaluate it where they need it)
static CompositeMap composite_of(const FramePlan* fp, bool paf, int cstride) {
    CompositeMap m;
    memset(&m, 0, sizeof(m));
    const int S = (int)fp->dims.size();
    m.n_scales = S;
    for (int i = 0; i < S; ++i) {
        CompositeScale& c = m.sc[i];
        const UpTables& t = fp->uptabs[i];
        c.src = paf ? fp->net->out_paf[i] : fp->net->out_heat[i];
        c.ho = fp->dims[i].ho;
        c.wo = fp->dims[i].wo;
        c.cstride = cstride;
        c.frame_stride = (size_t)c.ho * c.wo * cstride;
        c.xf = t.xf; c.xw = t.xw; c.yf = t.yf; c.yw = t.yw;
        c.ybf = t.ybf; c.ybr = t.ybr; c.ybw = t.ybw; c.yb_rs = t.yb_rs;
        c.l1 = (float)(t.l1 * 1.00001);
        c.sum_min = (float)(t.sum_min - 1e-5 * std::fabs(t.sum_min));
        c.sum_max = (float)(t.sum_max + 1e-5 * std::fabs(t.sum_max));
    }
    m.fused_ok = fp->fused_ok;
    return m;
}

// peaks -> grouping -> result copy for frames [f0, f0 + nf) of the batch.  mode 0: sigma-3 smoothing + NMS scored on
// the raw map (src/body.py:70-94); mode 1: NMS on the 5x5-blurred map scored with the blurred value (utilmx.py:230-241).
static void body_post_range(opb_session* s, FramePlan* fp, int f0, int nf, int H, int W) {
    cudaStream_t st = s->stream;
    const int mode = fp->key.mode >= 1 ? 1 : 0;
    OPB_CUDA(cudaMemsetAsync(fp->counters + (size_t)f0 * kCounterInts, 0, (size_t)nf * kCounterInts * sizeof(int), st));
    MapSource heat, paf;
    heat.frame_base = paf.frame_base = f0;
    if (fp->fused_ok) {
        heat.comp = composite_of(fp, false, 24);
    } else {
        if (f0 == 0) run_upsample(fp, false, fp->key.n, 19, 24, H, W, fp->heat_avg, st);
        heat.planar = fp->heat_avg;
        heat.planes_per_frame = 19;
    }
    paf.comp = composite_of(fp, true, 40);
    int peak_cap = 0, subset_cap = 0, pair_cap = 0;
    for (int f = f0; f < f0 + nf; ++f) {
        peak_cap = std::max(peak_cap, fp->post[f].pb.capacity);
        subset_cap = std::max(subset_cap, fp->post[f].lb.subset_capacity);
        pair_cap = std::max(pair_cap, fp->post[f].lb.pair_capacity);
    }
    find_peaks_launch(heat, nf, H, W, 18, mode, 0.1, fp->post_dev + f0, nullptr, fp->tile_mask, st);      // thre1: src/body.py:30, Batch_model.py:121
    s->prof.mark(st, "find_peaks");
    order_peaks_launch(fp->post_dev + f0, nf, peak_cap, 18, st);
    s->prof.mark(st, "order_peaks");
    paf_group_launch(paf, nf, H, W, fp->post_dev + f0, 0.05, subset_cap, pair_cap, peak_cap, st);               // thre2, src/body.py:31
    s->prof.mark(st, "paf_group");
    pack_results_launch(fp->post_dev + f0, nf, st);
    OPB_CUDA(cudaMemcpyAsync(s->host + f0, fp->results_dev + f0, (size_t)nf * sizeof(FrameResults), cudaMemcpyDeviceToHost, st));
    s->prof.mark(st, "d2h");
}

static void body_post_enqueue(opb_session* s, FramePlan* fp, int n, int H, int W) {
    body_post_range(s, fp, 0, n, H, W);
}

// A frame produced more peaks / scored limb pairs / connections / person rows than its buffers hold (the reference has
// no such limits): give that frame larger buffers, repeat its post-processing from the net outputs that are still on
// the device, and make the plan re-capture its graph.  Returns false when nothing can grow any further.
static bool grow_and_redo(opb_session* s, FramePlan* fp, int f, int appended, int status) {
    FramePost& bp = fp->post[f];
    int peak_cap = bp.pb.capacity, pair_cap = bp.lb.pair_capacity, conn_cap = bp.lb.conn_capacity;
    int subset_cap = bp.lb.subset_capacity;
    constexpr int kMaxPeaks = 1 << 18, kMaxPairs = 1 << 20, kMaxConn = 1 << 16, kMaxSubset = 1 << 16;      // 2^18 peaks: 64 KB of bitmaps in limb matching
    bool grew = false;
    if (appended > peak_cap && peak_cap < kMaxPeaks) {
        while (peak_cap < appended && peak_cap < kMaxPeaks) peak_cap *= 4;
        grew = true;
    }
    if ((status & kStPairOverflow) && pair_cap < kMaxPairs) {
        pair_cap *= 4;
        grew = true;
    }
    if ((status & kStConnOverflow) && conn_cap < kMaxConn) {
        conn_cap *= 4;
        grew = true;
    }
    if ((status & kStSubsetOverflow) && subset_cap < kMaxSubset) {        // beyond 1024 rows: global work rows
        subset_cap *= 4;
        grew = true;
    }
    if (!grew) return false;
    OPB_CUDA(cudaStreamSynchronize(s->stream));
    FramePost bigger;
    alloc_body_post(fp->pool, bigger, fp->counters + (size_t)f * kCounterInts, fp->results_dev + f, peak_cap, pair_cap,
                    conn_cap, subset_cap);
    bp = bigger;                                         // the old buffers stay in the plan's pool until it dies
    upload_post_table(fp, s->stream);
    if (fp->graph) {
        cudaGraphExecDestroy(fp->graph);
        fp->graph = nullptr;
    }
    if (fp->pose_graph) {
        cudaGraphExecDestroy(fp->pose_graph);
        fp->pose_graph = nullptr;
    }
    if (fp->batch_pose_graph) {
        cudaGraphExecDestroy(fp->batch_pose_graph);
        fp->batch_pose_graph = nullptr;
    }
    if (fp->every_graph) {
        cudaGraphExecDestroy(fp->every_graph);
        fp->every_graph = nullptr;
    }
    const bool prof = s->prof.on;
    s->prof.on = false;
    body_post_range(s, fp, f, 1, fp->key.H, fp->key.W);
    s->prof.on = prof;
    OPB_CUDA(cudaStreamSynchronize(s->stream));
    return true;
}

static void finish_submit(opb_session* s, FramePlan* fp) {
    OPB_CUDA(cudaEventRecord(s->done, s->stream));
    s->net->ctx->launches += fp->launches_per_frame;
}

static void body_submit(opb_session* s, const uint8_t* img, int where, int n, int H, int W, const double* scales, int ns) {
    OPB_REQUIRE(s->net->kind == OPB_NET_BODY, "session was created on a hand network");
    OPB_REQUIRE(n >= 1 && n <= 64, "1..64 frames per batch");
    OPB_CUDA(cudaSetDevice(s->net->ctx->device));
    FramePlan* fp = get_plan(s, n, H, W, scales, ns);
    ensure_host(s, n, 0);
    s->active = fp;
    s->n_frames = n;
    cudaStream_t st = s->stream;
    s->prof.reset();
    s->prof.mark(st, "start");
    upload_image(s, fp, img, where, (size_t)n * H * W * 3);
    s->prof.mark(st, "h2d");
    run_or_replay(s, fp, [&] {
        run_front(s, fp, n, H, W);
        body_post_enqueue(s, fp, n, H, W);
    });
    finish_submit(s, fp);
}

// float front end of the batched estimators: resize (body only) - 0.5, zero pad, bf16 HWC3 -> CNN
static void run_front_f32(opb_session* s, FramePlan* fp, int n, int H, int W) {
    cudaStream_t st = s->stream;
    const ScaleDims& d = fp->dims[0];
    const F32Taps& t = fp->f32taps[0];
    preprocess_f32_launch(fp->d_img, fp->key.mode == 2, n, H, W, fp->net->in_u8[0], d.h, d.w, d.hp, d.wp, t.xf, t.xc, t.yf, t.yc, st);
    s->prof.mark(st, "preprocess");
    fp->net->run(st, s->prof.on ? &s->prof : nullptr);
}

// Batch_body.__call__ (srcmx/Batch_model.py:142-204)
static void batch_body_submit(opb_session* s, const void* frames, bool u8, int where, int n, int H, int W, double g_scale) {
    OPB_REQUIRE(s->net->kind == OPB_NET_BODY, "session was created on a hand network");
    OPB_REQUIRE(n >= 1 && n <= 64, "1..64 frames per batch");
    OPB_REQUIRE(g_scale > 0, "scale must be positive");
    OPB_CUDA(cudaSetDevice(s->net->ctx->device));
    FramePlan* fp = get_plan(s, n, H, W, &g_scale, 1, u8 ? 2 : 1);
    ensure_host(s, n, 0);
    s->active = fp;
    s->n_frames = n;
    cudaStream_t st = s->stream;
    s->prof.reset();
    s->prof.mark(st, "start");
    upload_image(s, fp, (const uint8_t*)frames, where, (size_t)n * H * W * 3 * (u8 ? 1 : sizeof(float)));
    s->prof.mark(st, "h2d");
    run_or_replay(s, fp, [&] {
        run_front_f32(s, fp, n, H, W);
        body_post_enqueue(s, fp, n, H, W);              // 5x5 blur (utilmx.py:261-263) inside the peak kernel
    });
    finish_submit(s, fp);
}

// returns the first non-OK per-frame status (OPB_ERR_SUBSET_INDEX mirrors the reference's IndexError)
static int body_wait(opb_session* s, int* n_cand, int* n_subset, int* frame_status) {
    OPB_REQUIRE(s->active != nullptr, "no frame in flight");
    FramePlan* fp = s->active;
    OPB_CUDA(cudaEventSynchronize(s->done));
    s->results.assign(s->n_frames, FrameResult());
    int rc = OPB_OK;
    bool extra = false;
    for (int f = 0; f < s->n_frames; ++f) {
        HostResults* h = s->host + f;
        FramePost& bp = fp->post[f];
        FrameResult& r = s->results[f];
        int appended = h->counts[0];
        int status = h->counts[21];
        for (int attempt = 0; attempt < 12; ++attempt) {
            if (appended <= bp.pb.capacity && !(status & (kStPairOverflow | kStConnOverflow | kStSubsetOverflow))) break;
            if (!grow_and_redo(s, fp, f, appended, status)) break;
            appended = h->counts[0];
            status = h->counts[21];
        }
        if (appended > bp.pb.capacity)
            throw Error(OPB_ERR_CAPACITY, "more than " + std::to_string(bp.pb.capacity) + " heat-map peaks in one frame");
        if (status & (kStPairOverflow | kStConnOverflow | kStSubsetOverflow))
            throw Error(OPB_ERR_CAPACITY, "limb / person buffers overflowed (status " + std::to_string(status) + ")");
        r.n_cand = h->counts[19];            // part_begin[18] = total
        r.n_subset = h->counts[20];
        r.status = (status & kStIndexError) ? OPB_ERR_SUBSET_INDEX : OPB_OK;
        if (r.n_cand > kEagerCand) {
            r.cand_all.resize((size_t)r.n_cand * 4);
            OPB_CUDA(cudaMemcpyAsync(r.cand_all.data(), bp.pb.candidates, r.cand_all.size() * 8, cudaMemcpyDeviceToHost, s->stream));
            extra = true;
        }
        if (r.n_subset > kEagerSubset) {
            r.subset_all.resize((size_t)r.n_subset * 20);
            OPB_CUDA(cudaMemcpyAsync(r.subset_all.data(), bp.lb.subset, r.subset_all.size() * 8, cudaMemcpyDeviceToHost, s->stream));
            extra = true;
        }
        if (n_cand) n_cand[f] = r.n_cand;
        if (n_subset) n_subset[f] = r.n_subset;
        if (frame_status) frame_status[f] = r.status;
        if (r.status != OPB_OK && rc == OPB_OK) rc = r.status;
    }
    if (extra) OPB_CUDA(cudaStreamSynchronize(s->stream));
    if (rc == OPB_ERR_SUBSET_INDEX)
        set_last_error("list assignment index out of range (three subset rows match one connection, src/body.py:173)");
    return rc;
}

static void body_fetch(opb_session* s, int frame, double* candidate, int cand_rows, double* subset, int subset_rows) {
    OPB_REQUIRE(s->active && frame >= 0 && frame < (int)s->results.size(), "no finished frame with this index");
    const FrameResult& r = s->results[frame];
    if (cand_rows < r.n_cand || subset_rows < r.n_subset) throw Error(OPB_ERR_CAPACITY, "fetch buffers smaller than the result");
    if (r.n_cand) {
        OPB_REQUIRE(candidate != nullptr, "null candidate buffer");
        const double* src = r.cand_all.empty() ? s->host[frame].cand : r.cand_all.data();
        memcpy(candidate, src, (size_t)r.n_cand * 4 * sizeof(double));
    }
    if (r.n_subset) {
        OPB_REQUIRE(subset != nullptr, "null subset buffer");
        const double* src = r.subset_all.empty() ? s->host[frame].subset : r.subset_all.data();
        memcpy(subset, src, (size_t)r.n_subset * 20 * sizeof(double));
    }
}

static void hand_submit(opb_session* s, const uint8_t* img, int where, int n, int H, int W, const double* scales, int ns) {
    OPB_REQUIRE(s->net->kind == OPB_NET_HAND, "session was created on a body network");
    OPB_REQUIRE(n >= 1 && n <= 1024, "1..1024 crops per batch");
    OPB_CUDA(cudaSetDevice(s->net->ctx->device));
    FramePlan* fp = get_plan(s, n, H, W, scales, ns);
    ensure_host(s, 1, (size_t)n * 63);
    s->active = fp;
    s->hand_crops = n;
    s->hand_ragged = false;
    cudaStream_t st = s->stream;
    s->prof.reset();
    s->prof.mark(st, "start");
    upload_image(s, fp, img, where, (size_t)n * H * W * 3);
    s->prof.mark(st, "h2d");
    run_or_replay(s, fp, [&] {
        run_front(s, fp, n, H, W);
        run_upsample(fp, false, n, 22, 24, H, W, fp->heat_avg, st);
        s->prof.mark(st, "upsample_avg");
        hand_peaks_launch2(fp->heat_avg, n, 22, H, W, 0.03, fp->hb, nullptr, st);    // thre, src/hand.py:31
        s->prof.mark(st, "hand_peaks");
        OPB_CUDA(cudaMemcpyAsync(s->hand_host, fp->hb.peaks, (size_t)n * 63 * sizeof(double), cudaMemcpyDeviceToHost, st));
        s->prof.mark(st, "d2h");
    });
    finish_submit(s, fp);
}

// Batch_hand.__call__ (srcmx/Batch_model.py:366-406) on the crops already in the plan's input buffer: peaks of every
// crop in fp->hb.peaks
static void batch_hand_enqueue(opb_session* s, FramePlan* fp, int n, int H, int W) {
    cudaStream_t st = s->stream;
    run_front_f32(s, fp, n, H, W);
    run_upsample(fp, false, n, 22, 24, H, W, fp->heat_avg, st);                                    // x8 bicubic, :377
    s->prof.mark(st, "upsample_avg");
    blur5_planar_launch(fp->heat_avg, fp->blurred, n * 22, H, W, st);                                     // :378
    s->prof.mark(st, "blur5");
    hand_peaks_blurred_launch(fp->blurred, n, 22, H, W, 0.035f, fp->hb, st);                       // thre, :361
    s->prof.mark(st, "hand_peaks");
}

static void batch_hand_submit(opb_session* s, const void* crops, bool u8, int where, int n, int H, int W) {
    OPB_REQUIRE(s->net->kind == OPB_NET_HAND, "session was created on a body network");
    OPB_REQUIRE(n >= 1 && n <= 1024, "1..1024 crops per batch");
    OPB_CUDA(cudaSetDevice(s->net->ctx->device));
    const double one = 1.0;
    FramePlan* fp = get_plan(s, n, H, W, &one, 1, u8 ? 2 : 1);
    ensure_host(s, 1, (size_t)n * 63);
    s->active = fp;
    s->hand_crops = n;
    s->hand_ragged = false;
    cudaStream_t st = s->stream;
    s->prof.reset();
    s->prof.mark(st, "start");
    upload_image(s, fp, (const uint8_t*)crops, where, (size_t)n * H * W * 3 * (u8 ? 1 : sizeof(float)));
    s->prof.mark(st, "h2d");
    run_or_replay(s, fp, [&] {
        batch_hand_enqueue(s, fp, n, H, W);
        OPB_CUDA(cudaMemcpyAsync(s->hand_host, fp->hb.peaks, (size_t)n * 63 * sizeof(double), cudaMemcpyDeviceToHost, st));
        s->prof.mark(st, "d2h");
    });
    finish_submit(s, fp);
}

// ------------------------------------------------------------------------------------------------
// the batched hand job on the device: Batch_hand_extraction, srcmx/Batch_motion_Estimation.py:19-63
// ------------------------------------------------------------------------------------------------
// Tap tables of cv2.resize(crop, (boxsize, boxsize), INTER_CUBIC) for every crop side 1..wmax, in the RaggedTables layout
// of the pose pipeline with one scale (only the preprocess entries are filled: the upsample runs on boxsize-square maps).
static void build_track_tables(opb_session::HandTrack& t, int boxsize, int wmax) {
    TableSlab slab;
    std::vector<unsigned> index((size_t)(wmax + 1) * 5, 0u);
    for (int w = 1; w <= wmax; ++w) {
        const CubicTaps taps = hand_track_taps(w, boxsize);
        index[(size_t)w * 5 + 0] = (unsigned)(size_t)slab.add(taps.first);
        index[(size_t)w * 5 + 1] = (unsigned)(size_t)slab.add(u8_coefs(taps));
    }
    OPB_REQUIRE(slab.host.size() < (1ull << 32), "hand-track tables exceed 4 GB");
    t.table_pool.release();
    uint8_t* dev = (uint8_t*)t.table_pool.alloc(slab.host.size());
    OPB_CUDA(cudaMemcpy(dev, slab.host.data(), slab.host.size(), cudaMemcpyHostToDevice));
    t.tabs.slab = dev;
    t.tabs.index = t.table_pool.upload(index);
    t.tabs.n_scales = 1;
    t.tabs.wmax = wmax;
    t.boxsize = boxsize;
    ++t.gen;
}
// the hand session's HandTrack with tables for `boxsize` and crops of up to wmax pixels (nothing may still use them)
static opb_session::HandTrack& track_with_tables(opb_session* s, int boxsize, int wmax) {
    if (!s->track) s->track = std::make_unique<opb_session::HandTrack>();
    opb_session::HandTrack& t = *s->track;
    if (t.boxsize != boxsize || t.tabs.wmax < wmax) build_track_tables(t, boxsize, wmax);
    return t;
}

static void hand_track_submit(opb_session* s, const uint8_t* frames, int where, int n, int H, int W, const double* poses,
                              int boxsize) {
    OPB_REQUIRE(s->net->kind == OPB_NET_HAND, "session was created on a body network");
    OPB_REQUIRE(n >= 1 && 2 * n <= 1024, "1..512 frames per batch (two crops each)");
    OPB_REQUIRE(H >= 1 && W >= 1, "empty frame");
    OPB_REQUIRE(boxsize >= 8 && boxsize % 8 == 0, "boxsize must be a positive multiple of 8 (srcmx/Batch_model.py:377)");
    OPB_CUDA(cudaSetDevice(s->net->ctx->device));
    cudaStream_t st = s->stream;
    OPB_CUDA(cudaStreamSynchronize(st));          // the pinned buffers and the tables may still serve the previous batch
    opb_session::HandTrack& t = track_with_tables(s, boxsize, std::min(H, W));
    if (t.frames < n) {
        t.pool.release();
        if (t.poses_host) cudaFreeHost(t.poses_host);
        if (t.mats_host) cudaFreeHost(t.mats_host);
        t.poses_host = t.mats_host = nullptr;
        t.frames = 0;
        t.poses = t.pool.alloc_t<double>((size_t)n * 54);
        t.boxes = t.pool.alloc_t<HandBox>((size_t)n * 2);
        t.mats = t.pool.alloc_t<double>((size_t)n * 126);
        OPB_CUDA(cudaMallocHost((void**)&t.poses_host, (size_t)n * 54 * sizeof(double)));
        OPB_CUDA(cudaMallocHost((void**)&t.mats_host, (size_t)n * 126 * sizeof(double)));
        t.frames = n;
        ++t.gen;
    }
    const size_t bytes = (size_t)n * H * W * 3;
    if (t.frame_bytes < bytes) {
        t.frame_pool.release();
        t.frames_dev = (uint8_t*)t.frame_pool.alloc(bytes);
        t.frame_bytes = bytes;
        ++t.gen;
    }
    if (t.H != H || t.W != W) ++t.gen;           // the captured launches carry the frame size
    t.H = H;
    t.W = W;
    t.n = n;
    memcpy(t.poses_host, poses, (size_t)n * 54 * sizeof(double));
    // the crops go straight into the input buffer of the uint8 Batch_hand plan of 2n boxsize-square crops
    const int slots = 2 * n;
    const double one = 1.0;
    FramePlan* fp = get_plan(s, slots, boxsize, boxsize, &one, 1, 2);
    s->active = fp;
    s->hand_crops = slots;
    s->hand_ragged = false;
    t.plan = fp;
    s->prof.reset();
    upload_bytes(s, t.frames_dev, frames, where, bytes);
    const uint64_t gen = (s->buffer_gen << 32) ^ t.gen;
    run_or_replay_slot(s, GraphSlot{fp->track_graph, fp->track_gen, fp->track_uses}, gen, [&] {
        OPB_CUDA(cudaMemcpyAsync(t.poses, t.poses_host, (size_t)n * 54 * sizeof(double), cudaMemcpyHostToDevice, st));
        hand_track_boxes_launch(t.poses, n, H, W, t.boxes, st);
        preprocess_ragged_launch(t.frames_dev, H, W, t.boxes, slots, fp->d_img, boxsize, 0, t.tabs, st);
        batch_hand_enqueue(s, fp, slots, boxsize, boxsize);
        hand_track_finish_launch(t.boxes, fp->hb.peaks, n, boxsize, t.mats, 126, st);
        OPB_CUDA(cudaMemcpyAsync(t.mats_host, t.mats, (size_t)n * 126 * sizeof(double), cudaMemcpyDeviceToHost, st));
    });
    OPB_CUDA(cudaEventRecord(s->done, st));
    s->net->ctx->launches += 3 /* boxes, crops, finish */ + fp->launches_per_frame;
}


// ------------------------------------------------------------------------------------------------
// per-frame caller on the device: MotionData_every_frame(mode='bodyhand'), srcmx/MotionEstimation.py:126-216
// ------------------------------------------------------------------------------------------------
// Tap tables for every square crop of side 1..wmax at the hand estimator's scales, built with the same host functions
// as the single-size path (so a ragged slot is processed exactly like Hand()(crop) would process that crop).
static std::unique_ptr<opb_session::Ragged> build_ragged_tables(const double* scales, int ns, int wmax) {
    auto r = std::make_unique<opb_session::Ragged>();
    r->scales.assign(scales, scales + ns);
    TableSlab slab;
    std::vector<unsigned> index((size_t)(wmax + 1) * ns * 5, 0u);
    r->net_side.assign(ns, 0);
    for (int w = 1; w <= wmax; ++w)
        for (int s = 0; s < ns; ++s) {
            const ScaleDims d = scale_dims(w, w, scales[s]);
            OPB_REQUIRE(d.h == d.w && d.hp == d.h, "hand scales must give square net inputs that are multiples of 8");
            if (r->net_side[s] == 0) r->net_side[s] = d.hp;
            OPB_REQUIRE(r->net_side[s] == d.hp, "the net input side must not depend on the crop size (boxsize / crop * crop)");
            const U8Taps u = make_u8_taps(slab, w, w, d);
            std::vector<int> fx;
            std::vector<float> wx;
            composite_taps(d.wo, d.w, w, fx, wx);
            std::vector<float> wy(wx);
            for (auto& v : wy) v = v / (float)ns;                  // same fold as make_up_tables
            unsigned* e = &index[((size_t)w * ns + s) * 5];
            e[0] = (unsigned)(size_t)u.xf;
            e[1] = (unsigned)(size_t)u.xc;
            e[2] = (unsigned)(size_t)slab.add(fx);
            e[3] = (unsigned)(size_t)slab.add(wx);
            e[4] = (unsigned)(size_t)slab.add(wy);
        }
    OPB_REQUIRE(slab.host.size() < (1ull << 32), "ragged tables exceed 4 GB");
    uint8_t* dev = (uint8_t*)r->pool.alloc(slab.host.size());
    OPB_CUDA(cudaMemcpy(dev, slab.host.data(), slab.host.size(), cudaMemcpyHostToDevice));
    r->tabs.slab = dev;
    r->tabs.index = r->pool.upload(index);
    r->tabs.n_scales = ns;
    r->tabs.wmax = wmax;
    return r;
}

// the hand session's ragged tables cover every crop of an H x W frame at these scales; returns their crop side limit, the
// plane pitch of the ragged buffers
static int ensure_ragged_tables(opb_session* bs, opb_session* hs, int H, int W, const double* hscales, int nhs) {
    const int wmax = std::min(H, W);
    if (!hs->ragged || hs->ragged->tabs.wmax < wmax || hs->ragged->scales != std::vector<double>(hscales, hscales + nhs)) {
        OPB_CUDA(cudaStreamSynchronize(bs->stream));
        hs->ragged = build_ragged_tables(hscales, nhs, wmax);
    }
    return hs->ragged->tabs.wmax;
}

// per-batch [n][60][3] records, hand boxes and their pinned host copy on a body session, grown to the largest batch seen
static void ensure_pose_buffers(opb_session* bs, int n) {
    if (bs->pose && bs->pose->frames >= n) return;
    OPB_CUDA(cudaStreamSynchronize(bs->stream));
    auto pb = std::make_unique<opb_session::PoseBuffers>();
    pb->frames = n;
    pb->pose = pb->pool.alloc_t<double>((size_t)n * 180);
    pb->boxes = pb->pool.alloc_t<HandBox>((size_t)n * 2);
    pb->dims = pb->pool.alloc_t<int>((size_t)n * 2);
    pb->fixed = pb->pool.alloc_t<int>((size_t)n * 6);
    OPB_CUDA(cudaMallocHost((void**)&pb->host, (size_t)n * 180 * sizeof(double)));
    OPB_CUDA(cudaMallocHost((void**)&pb->fixed_host, (size_t)n * 6 * sizeof(int)));
    bs->pose = std::move(pb);
}

// Hand on `slots` boxes (dims: side of each valid box, else 0) of the frames `fp` holds, as one ragged batch on the hand
// plan `hp` of hs: crops cut -- the left ones mirrored -- from the frames -> hand CNN -> ragged post-processing, the
// key points of slot i at hp->hb.peaks + i * 63
static void ragged_hand_net_post(cudaStream_t st, const opb_session::Ragged& rg, FramePlan* hp, const HandBox* boxes,
                                 const int* dims, int slots);
static void ragged_hand_enqueue(cudaStream_t st, opb_session* hs, FramePlan* fp, FramePlan* hp, const HandBox* boxes,
                                const int* dims, int slots) {
    const opb_session::Ragged& rg = *hs->ragged;
    for (int s = 0; s < rg.tabs.n_scales; ++s)
        preprocess_ragged_launch(fp->d_img, fp->key.H, fp->key.W, boxes, slots, hp->net->in_u8[s], rg.net_side[s], s, rg.tabs, st);
    ragged_hand_net_post(st, rg, hp, boxes, dims, slots);
}
// the rest of a ragged hand batch once every slot's crop is resized into the net inputs of hp
static void ragged_hand_net_post(cudaStream_t st, const opb_session::Ragged& rg, FramePlan* hp, const HandBox* boxes,
                                 const int* dims, int slots) {
    const int tw = rg.tabs.wmax, nhs = rg.tabs.n_scales;
    const float* src[kMaxScales];
    int ho[kMaxScales], wo[kMaxScales];
    for (int s = 0; s < nhs; ++s) {
        src[s] = hp->net->out_heat[s];
        ho[s] = wo[s] = rg.net_side[s] / 8;
    }
    hp->net->run(st, nullptr);
    upsample_ragged_launch(src, ho, wo, nhs, 24, 22, boxes, slots, rg.tabs, tw, hp->up_scratch, hp->heat_avg, st);
    hand_peaks_ragged_launch(hp->heat_avg, slots, 22, dims, tw, 0.03, hp->hb, st);      // thre, src/hand.py:31
}

// Hand()(crop) for every crop of a list of square crops of any sides, as one ragged batch: crop i is the dense
// sides[i] x sides[i] x 3 image at bytes [offsets[i], offsets[i + 1]) of `packed`.  The crops are uploaded as they are
// into the input arena; the packed form of the ragged crop kernel resizes each one with the tables of its own side, and
// from there on the batch is the hand half of the pose pipeline (one CNN plan per crop count and scales, upsample,
// Gaussian, components and selection at each crop's own size).
static uint64_t gen_key(std::initializer_list<uint64_t> parts);
static void hand_submit_ragged(opb_session* s, const uint8_t* packed, const size_t* offsets, int where, int n,
                               const int* sides, const double* scales, int ns) {
    OPB_REQUIRE(s->net->kind == OPB_NET_HAND, "session was created on a body network");
    OPB_REQUIRE(n >= 1 && n <= 1024, "1..1024 crops per batch");
    OPB_REQUIRE(ns >= 1 && ns <= kMaxScales, "scale_search must hold 1..8 entries");
    OPB_REQUIRE(offsets[0] == 0, "offsets[0] must be 0 (the crops are packed back to back)");
    int wmax = 0;
    for (int i = 0; i < n; ++i) {
        OPB_REQUIRE(sides[i] >= 1, "empty crop (the reference divides by oriImg.shape[0], src/hand.py:32)");
        OPB_REQUIRE(offsets[i + 1] >= offsets[i] && offsets[i + 1] - offsets[i] == (size_t)sides[i] * sides[i] * 3,
                    "offsets[i + 1] - offsets[i] must be sides[i] * sides[i] * 3 bytes (crop " + std::to_string(i) + ")");
        wmax = std::max(wmax, sides[i]);
    }
    OPB_CUDA(cudaSetDevice(s->net->ctx->device));
    cudaStream_t st = s->stream;
    OPB_CUDA(cudaStreamSynchronize(st));          // the pinned crop list and the tables may still serve the previous batch
    const std::vector<double> sc(scales, scales + ns);
    if (!s->crop_tables || s->crop_tables->tabs.wmax < wmax || s->crop_tables->scales != sc)
        s->crop_tables = build_ragged_tables(scales, ns, wmax);
    const opb_session::Ragged& rg = *s->crop_tables;
    const int tw = rg.tabs.wmax;
    if (!s->crop_list || s->crop_list->cap < n) {
        auto cl = std::make_unique<opb_session::CropList>();
        cl->boxes = cl->pool.alloc_t<HandBox>(n);
        cl->sides = cl->pool.alloc_t<int>(n);
        cl->offsets = cl->pool.alloc_t<size_t>(n);
        OPB_CUDA(cudaMallocHost((void**)&cl->boxes_host, (size_t)n * sizeof(HandBox)));
        OPB_CUDA(cudaMallocHost((void**)&cl->sides_host, (size_t)n * sizeof(int)));
        OPB_CUDA(cudaMallocHost((void**)&cl->offsets_host, (size_t)n * sizeof(size_t)));
        cl->cap = n;
        s->crop_list = std::move(cl);
    }
    opb_session::CropList& cl = *s->crop_list;
    for (int i = 0; i < n; ++i) {
        cl.boxes_host[i] = HandBox{i, 0, 0, sides[i], 0, 1};
        cl.sides_host[i] = sides[i];
        cl.offsets_host[i] = offsets[i];
    }
    // the frame plan of n crops of the table side: its arenas hold n tw-square crops (more than the packed list needs)
    // and its CNN plan is the one every n-crop batch of these scales shares
    FramePlan* fp = get_plan(s, n, tw, tw, scales, ns);
    ensure_host(s, 1, (size_t)n * 63);
    s->active = fp;
    s->hand_crops = n;
    s->hand_ragged = true;
    s->prof.reset();
    upload_bytes(s, fp->d_img, packed, where, offsets[n]);
    const uint64_t gen = gen_key({s->buffer_gen, (uint64_t)(uintptr_t)cl.boxes, (uint64_t)(uintptr_t)rg.tabs.slab,
                                  (uint64_t)(uintptr_t)rg.tabs.index});
    run_or_replay_slot(s, GraphSlot{fp->crops_graph, fp->crops_gen, fp->crops_uses}, gen, [&] {
        OPB_CUDA(cudaMemcpyAsync(cl.boxes, cl.boxes_host, (size_t)n * sizeof(HandBox), cudaMemcpyHostToDevice, st));
        OPB_CUDA(cudaMemcpyAsync(cl.sides, cl.sides_host, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, st));
        OPB_CUDA(cudaMemcpyAsync(cl.offsets, cl.offsets_host, (size_t)n * sizeof(size_t), cudaMemcpyHostToDevice, st));
        for (int i = 0; i < ns; ++i)
            preprocess_packed_launch(fp->d_img, cl.offsets, cl.boxes, n, fp->net->in_u8[i], rg.net_side[i], i, rg.tabs, st);
        ragged_hand_net_post(st, rg, fp, cl.boxes, cl.sides, n);
        OPB_CUDA(cudaMemcpyAsync(s->hand_host, fp->hb.peaks, (size_t)n * 63 * sizeof(double), cudaMemcpyDeviceToHost, st));
    });
    OPB_CUDA(cudaEventRecord(s->done, st));
    s->net->ctx->launches += ns + fp->net->kernel_launches + (ns + 1) + 6;
}

// the hand half of the pose pipeline, on the body session's stream: boxes from the body results (or the fixed ones already
// in the pinned buffer), ragged crops -> hand CNN -> ragged post-processing -> PoseMat -> pinned host buffer
static void pose_hand_enqueue(opb_session* bs, opb_session* hs, FramePlan* fp, FramePlan* hp, int n, int H, int W, bool fixed) {
    cudaStream_t st = bs->stream;
    if (fixed)
        OPB_CUDA(cudaMemcpyAsync(bs->pose->fixed, bs->pose->fixed_host, (size_t)n * 6 * sizeof(int), cudaMemcpyHostToDevice, st));
    pose_select_launch(fp->post_dev, n, H, W, fixed ? bs->pose->fixed : nullptr, bs->pose->pose, bs->pose->boxes, bs->pose->dims, st);
    ragged_hand_enqueue(st, hs, fp, hp, bs->pose->boxes, bs->pose->dims, 2 * n);
    pose_finish_launch(bs->pose->boxes, hp->hb.peaks, n, bs->pose->pose, st);
    OPB_CUDA(cudaMemcpyAsync(bs->pose->host, bs->pose->pose, (size_t)n * 180 * sizeof(double), cudaMemcpyDeviceToHost, st));
}

static void pose_submit(opb_session* bs, opb_session* hs, const uint8_t* imgs, int where, int n, int H, int W,
                        const double* bscales, int nbs, const double* hscales, int nhs, const int* fixed_boxes) {
    OPB_REQUIRE(bs->net->kind == OPB_NET_BODY && hs->net->kind == OPB_NET_HAND, "pose: a body session and a hand session");
    OPB_REQUIRE(bs->net->ctx == hs->net->ctx, "pose: both networks must live on the same context");
    OPB_REQUIRE(n >= 1 && n <= 64, "1..64 frames per batch");
    OPB_CUDA(cudaSetDevice(bs->net->ctx->device));
    const int slots = 2 * n;
    const int tw = ensure_ragged_tables(bs, hs, H, W, hscales, nhs);
    ensure_pose_buffers(bs, n);
    // body part: as opb_body_submit_batch
    FramePlan* fp = get_plan(bs, n, H, W, bscales, nbs);
    ensure_host(bs, n, 0);
    bs->active = fp;
    bs->n_frames = n;
    bs->pose_hand = hs;
    bs->batch_pose_box = 0;
    bs->every_batch = false;
    cudaStream_t st = bs->stream;
    upload_image(bs, fp, imgs, where, (size_t)n * H * W * 3);
    // hand part on the same stream, with the hand session's CNN plan and work buffers (sized for the largest crop)
    OPB_CUDA(cudaStreamSynchronize(hs->stream));               // nothing of the hand session's own stream may still use them
    FramePlan* hp = get_plan(hs, slots, tw, tw, hscales, nhs);
    hs->active = hp;
    hs->hand_crops = slots;
    hs->hand_ragged = false;
    int* fixed_dev = nullptr;
    if (fixed_boxes) {
        OPB_CUDA(cudaStreamSynchronize(st));                   // the pinned copy of the previous batch's boxes is free
        memcpy(bs->pose->fixed_host, fixed_boxes, (size_t)n * 6 * sizeof(int));
        fixed_dev = bs->pose->fixed;
    }
    // everything between the frame upload and the PoseMat copy is one launch sequence on one stream: replayed as a CUDA
    // graph from the third use on (re-captured when a buffer of either session, the hand plan or the box source changed)
    const uint64_t gen = bs->buffer_gen * 1000003ull + hs->buffer_gen * 7919ull + (uint64_t)(uintptr_t)hp +
                         (uint64_t)(uintptr_t)hs->ragged->tabs.slab + (fixed_dev ? 1 : 0);
    bs->pose_hand_scales.assign(hscales, hscales + nhs);
    bs->pose_fixed = fixed_dev != nullptr;
    run_or_replay_slot(bs, GraphSlot{fp->pose_graph, fp->pose_gen, fp->pose_uses}, gen, [&] {
        run_front(bs, fp, n, H, W);
        body_post_enqueue(bs, fp, n, H, W);
        pose_hand_enqueue(bs, hs, fp, hp, n, H, W, fixed_dev != nullptr);
    });
    OPB_CUDA(cudaEventRecord(bs->done, st));
    bs->net->ctx->launches += fp->launches_per_frame + nhs + hp->net->kernel_launches + (nhs + 1) + 6 + 2;
}

// the overflow check of a pose batch after its body results arrived: a frame that overflowed its peak / pair / connection
// / person buffers gets larger ones and its body post-processing is repeated (like opb_body_wait_batch; `grew` tells the
// caller to repeat the hand half of the batch).  Fills frame_status (optional) and returns the first non-OK status.
static int pose_batch_status(opb_session* bs, int* frame_status, bool& grew) {
    int rc = OPB_OK;
    OPB_CUDA(cudaEventSynchronize(bs->done));
    FramePlan* fp = bs->active;
    for (int f = 0; f < bs->n_frames; ++f) {
        const HostResults* h = bs->host + f;
        for (int attempt = 0; attempt < 12; ++attempt) {
            const FramePost& bp = fp->post[f];
            if (h->counts[0] <= bp.pb.capacity && !(h->counts[21] & (kStPairOverflow | kStConnOverflow | kStSubsetOverflow))) break;
            if (!grow_and_redo(bs, fp, f, h->counts[0], h->counts[21])) break;
            grew = true;
        }
        const int status = h->counts[21];
        if (h->counts[0] > fp->post[f].pb.capacity || (status & (kStPairOverflow | kStConnOverflow | kStSubsetOverflow)))
            throw Error(OPB_ERR_CAPACITY, "a frame overflowed the body result buffers (status " + std::to_string(status) + ")");
        const int st = (status & kStIndexError) ? OPB_ERR_SUBSET_INDEX : OPB_OK;
        if (frame_status) frame_status[f] = st;
        if (st != OPB_OK && rc == OPB_OK) rc = st;
    }
    if (rc == OPB_ERR_SUBSET_INDEX)
        set_last_error("list assignment index out of range (three subset rows match one connection, src/body.py:173)");
    return rc;
}

// ------------------------------------------------------------------------------------------------
// the one-pass body + hand job: Batch_body_extraction and Batch_hand_extraction (srcmx/Batch_motion_Estimation.py:19-112)
// on one upload of the decoded frames
// ------------------------------------------------------------------------------------------------
// The hand half, on the body session's stream: person, body rows and both hand boxes from the Batch_body results, both
// crops cut from the frames still in the body plan's input buffer into the uint8 Batch_hand plan `hp` of the hand session,
// Batch_hand on all 2n crops, HandMat into rows 18-59 of the records, one copy of the records into pinned host memory.
static void batch_pose_hand_enqueue(opb_session* bs, opb_session* hs, FramePlan* fp, FramePlan* hp, int n, int boxsize) {
    cudaStream_t st = bs->stream;
    const int H = fp->key.H, W = fp->key.W, slots = 2 * n;
    const opb_session::PoseBuffers& pb = *bs->pose;
    batch_pose_select_launch(fp->post_dev, n, H, W, pb.pose, pb.boxes, st);
    preprocess_ragged_launch(fp->d_img, H, W, pb.boxes, slots, hp->d_img, boxsize, 0, hs->track->tabs, st);
    batch_hand_enqueue(bs, hp, slots, boxsize, boxsize);        // bs only lends its stream and profiler
    hand_track_finish_launch(pb.boxes, hp->hb.peaks, n, boxsize, pb.pose + 54, 180, st);
    OPB_CUDA(cudaMemcpyAsync(pb.host, pb.pose, (size_t)n * 180 * sizeof(double), cudaMemcpyDeviceToHost, st));
}

static uint64_t gen_key(std::initializer_list<uint64_t> parts) {      // FNV-1a over the words
    uint64_t h = 14695981039346656037ull;
    for (uint64_t v : parts) h = (h ^ v) * 1099511628211ull;
    return h;
}

static void batch_pose_submit(opb_session* bs, opb_session* hs, const uint8_t* frames, int where, int n, int H, int W,
                              double g_scale, int boxsize) {
    OPB_REQUIRE(bs->net->kind == OPB_NET_BODY && hs->net->kind == OPB_NET_HAND,
                "batch pose: a body session and a hand session");
    OPB_REQUIRE(bs->net->ctx == hs->net->ctx, "batch pose: both networks must live on the same context");
    OPB_REQUIRE(n >= 1 && n <= 64, "1..64 frames per batch");
    OPB_REQUIRE(H >= 1 && W >= 1, "empty frame");
    OPB_REQUIRE(g_scale > 0, "scale must be positive");
    OPB_REQUIRE(boxsize >= 8 && boxsize % 8 == 0, "boxsize must be a positive multiple of 8 (srcmx/Batch_model.py:377)");
    OPB_CUDA(cudaSetDevice(bs->net->ctx->device));
    cudaStream_t st = bs->stream;
    // the records, boxes and crop tables may still serve the previous batch of this pair, the hand plan work of the
    // hand session's own stream
    OPB_CUDA(cudaStreamSynchronize(st));
    OPB_CUDA(cudaStreamSynchronize(hs->stream));
    ensure_pose_buffers(bs, n);
    opb_session::HandTrack& t = track_with_tables(hs, boxsize, std::min(H, W));
    FramePlan* fp = get_plan(bs, n, H, W, &g_scale, 1, 2);          // Batch_body on uint8 frames
    ensure_host(bs, n, 0);
    bs->active = fp;
    bs->n_frames = n;
    bs->pose_hand = hs;
    bs->batch_pose_box = boxsize;
    bs->every_batch = false;
    const double one = 1.0;
    FramePlan* hp = get_plan(hs, 2 * n, boxsize, boxsize, &one, 1, 2);      // uint8 Batch_hand on 2n crops
    hs->active = hp;
    hs->hand_crops = 2 * n;
    hs->hand_ragged = false;
    t.plan = hp;
    bs->prof.reset();
    bs->prof.mark(st, "start");
    upload_image(bs, fp, frames, where, (size_t)n * H * W * 3);
    bs->prof.mark(st, "h2d");
    // one launch sequence from the uploaded frames to the records copy, replayed as a CUDA graph from the third use on;
    // re-captured when a buffer of either session, the hand plan, the crop tables, the records or the frame size change
    const opb_session::PoseBuffers& pb = *bs->pose;
    const uint64_t gen = gen_key({bs->buffer_gen, hs->buffer_gen, (uint64_t)(uintptr_t)hp, t.gen,
                                  (uint64_t)(uintptr_t)pb.pose, (uint64_t)(uintptr_t)pb.boxes, (uint64_t)(uintptr_t)pb.host,
                                  (uint64_t)H, (uint64_t)W, (uint64_t)boxsize});
    run_or_replay_slot(bs, GraphSlot{fp->batch_pose_graph, fp->batch_pose_gen, fp->batch_pose_uses}, gen, [&] {
        run_front_f32(bs, fp, n, H, W);
        body_post_enqueue(bs, fp, n, H, W);
        batch_pose_hand_enqueue(bs, hs, fp, hp, n, boxsize);
    });
    OPB_CUDA(cudaEventRecord(bs->done, st));
    bs->net->ctx->launches += fp->launches_per_frame + 3 /* select, crops, finish */ + hp->launches_per_frame;
}

// ------------------------------------------------------------------------------------------------
// every person of every frame: Body, util.handDetect on every subset row (src/util.py:133-201), Hand on every box --
// the caller's host loop on the reference's Body / Hand, with the PoseMat arithmetic of MotionEstimation.py:185-194
// ------------------------------------------------------------------------------------------------
// Hand slots per chunk.  The ragged hand buffers grow with slots x min(H, W)^2; 8 slots are half of what
// opb_pose_submit_batch holds at 8 frames (16 slots).  The CNN runs on every slot of a chunk, the empty ones of the
// last chunk too, so a smaller chunk wastes less on a batch with few hands.
constexpr int kEveryChunk = 8;
// Crops per chunk of the batched estimators' every-person path (opb_batch_pose_every_*): boxsize-square crops through a
// uint8 Batch_hand plan.  Measured on a B200 at 16, 32 and 64 (DESIGN.md section 7, N2): 16 is 3.5 % slower, 64 only
// 0.3 % faster than 32 but doubles the plan's activations and the CNN slots wasted in a batch's last partial chunk.
constexpr int kBatchEveryChunk = 32;
constexpr int kEveryChunkSlots = kEveryChunk > kBatchEveryChunk ? kEveryChunk : kBatchEveryChunk;

// records and box list for `persons` persons (grown by doubling; OPB_TEST_SMALL_BUFFERS starts tiny so that tests reach
// the growth path of opb_pose_every_wait)
static void ensure_every_buffers(opb_session* bs, int persons) {
    if (bs->every && bs->every->cap >= persons) return;
    static const bool tiny = getenv("OPB_TEST_SMALL_BUFFERS") != nullptr;
    int cap = bs->every ? 2 * bs->every->cap : (tiny ? 2 : 512);
    while (cap < persons) cap *= 2;
    OPB_CUDA(cudaStreamSynchronize(bs->stream));
    auto e = std::make_unique<opb_session::EveryBuffers>();
    e->cap = cap;
    e->gen = ++bs->every_allocs;
    e->records = e->pool.alloc_t<double>((size_t)cap * 180);
    e->list = e->pool.alloc_t<HandBox>((size_t)cap * 2);
    e->list_rec = e->pool.alloc_t<int>((size_t)cap * 2);
    e->counts = e->pool.alloc_t<int>(kEveryCounts, true);
    e->chunk_boxes = e->pool.alloc_t<HandBox>(kEveryChunkSlots);
    e->chunk_dims = e->pool.alloc_t<int>(kEveryChunkSlots);
    e->chunk_rec = e->pool.alloc_t<int>(kEveryChunkSlots);
    OPB_CUDA(cudaMallocHost((void**)&e->records_host, (size_t)cap * 180 * sizeof(double)));
    OPB_CUDA(cudaMallocHost((void**)&e->counts_host, kEveryCounts * sizeof(int)));
    e->ids = e->pool.alloc_t<int>(cap);
    OPB_CUDA(cudaMallocHost((void**)&e->ids_host, (size_t)cap * sizeof(int)));
    bs->every = std::move(e);
}

// rows and boxes of every person from the body results of the batch (the batched estimators' box rule for an
// opb_batch_pose_every batch); the counts to pinned memory
static void every_rows_enqueue(opb_session* bs, FramePlan* fp, int n) {
    opb_session::EveryBuffers& e = *bs->every;
    every_rows_launch(fp->post_dev, n, fp->key.H, fp->key.W, e.cap, e.records, e.list, e.list_rec, e.counts,
                      bs->batch_pose_box != 0, bs->stream);
    OPB_CUDA(cudaMemcpyAsync(e.counts_host, e.counts, kEveryCounts * sizeof(int), cudaMemcpyDeviceToHost, bs->stream));
}

// one chunk of the hand half: the next kEveryChunk boxes of the list (the cursor lives on the device, so the same launch
// sequence -- one CUDA graph -- serves every chunk of every batch), Hand on them, key points into their records
static void every_chunk_enqueue(opb_session* bs, opb_session* hs, FramePlan* fp, FramePlan* hp) {
    cudaStream_t st = bs->stream;
    opb_session::EveryBuffers& e = *bs->every;
    every_stage_launch(e.list, e.list_rec, e.counts, kEveryChunk, e.chunk_boxes, e.chunk_dims, e.chunk_rec, st);
    ragged_hand_enqueue(st, hs, fp, hp, e.chunk_boxes, e.chunk_dims, kEveryChunk);
    every_finish_launch(e.chunk_boxes, e.chunk_rec, hp->hb.peaks, kEveryChunk, e.records, e.counts, st);
}

static void every_submit(opb_session* bs, opb_session* hs, const uint8_t* imgs, int where, int n, int H, int W,
                         const double* bscales, int nbs, const double* hscales, int nhs) {
    OPB_REQUIRE(bs->net->kind == OPB_NET_BODY && hs->net->kind == OPB_NET_HAND, "every person: a body session and a hand session");
    OPB_REQUIRE(bs->net->ctx == hs->net->ctx, "every person: both networks must live on the same context");
    OPB_REQUIRE(n >= 1 && n <= 64, "1..64 frames per batch");
    OPB_REQUIRE(H >= 1 && W >= 1, "empty frame");
    OPB_CUDA(cudaSetDevice(bs->net->ctx->device));
    cudaStream_t st = bs->stream;
    const int tw = ensure_ragged_tables(bs, hs, H, W, hscales, nhs);
    ensure_every_buffers(bs, 0);
    FramePlan* fp = get_plan(bs, n, H, W, bscales, nbs);
    ensure_host(bs, n, 0);
    bs->active = fp;
    bs->n_frames = n;
    bs->pose_hand = hs;
    bs->batch_pose_box = 0;
    bs->every_batch = true;
    bs->every_persons = -1;
    bs->every_linked = false;
    upload_image(bs, fp, imgs, where, (size_t)n * H * W * 3);
    // the hand plan of the chunks, with the hand session's work buffers sized for the largest crop
    OPB_CUDA(cudaStreamSynchronize(hs->stream));
    FramePlan* hp = get_plan(hs, kEveryChunk, tw, tw, hscales, nhs);
    hs->active = hp;
    hs->hand_crops = kEveryChunk;
    hs->hand_ragged = false;
    const uint64_t gen = gen_key({bs->buffer_gen, bs->every->gen});
    run_or_replay_slot(bs, GraphSlot{fp->every_graph, fp->every_gen, fp->every_uses}, gen, [&] {
        run_front(bs, fp, n, H, W);
        body_post_enqueue(bs, fp, n, H, W);
        every_rows_enqueue(bs, fp, n);
    });
    OPB_CUDA(cudaEventRecord(bs->done, st));
    bs->net->ctx->launches += fp->launches_per_frame + 1;
}

// ------------------------------------------------------------------------------------------------
// every person on the batched estimators: Batch_body, the body rows of every subset row and both hand crops of every
// person as Batch_hand_extraction derives them from a saved MotionMat row (grey crops for missing hands), Batch_hand on
// every crop, _box_to_roi into the records.  The waits, fetches, growth and tracking are every_wait's.
// ------------------------------------------------------------------------------------------------
// one chunk of the hand half: the next kBatchEveryChunk slots of the list, their crops cut from the frames still in the
// Batch_body plan's input buffer into the uint8 Batch_hand plan hp, Batch_hand on all of them, key points into records
static void batch_every_chunk_enqueue(opb_session* bs, opb_session* hs, FramePlan* fp, FramePlan* hp, int boxsize) {
    cudaStream_t st = bs->stream;
    opb_session::EveryBuffers& e = *bs->every;
    const int C = kBatchEveryChunk;
    every_stage_launch(e.list, e.list_rec, e.counts, C, e.chunk_boxes, e.chunk_dims, e.chunk_rec, st);
    preprocess_ragged_launch(fp->d_img, fp->key.H, fp->key.W, e.chunk_boxes, C, hp->d_img, boxsize, 0, hs->track->tabs, st);
    batch_hand_enqueue(bs, hp, C, boxsize, boxsize);            // bs only lends its stream and profiler
    batch_every_finish_launch(e.chunk_boxes, e.chunk_rec, hp->hb.peaks, C, boxsize, e.records, e.counts, st);
}

static void batch_every_submit(opb_session* bs, opb_session* hs, const uint8_t* frames, int where, int n, int H, int W,
                               double g_scale, int boxsize) {
    OPB_REQUIRE(bs->net->kind == OPB_NET_BODY && hs->net->kind == OPB_NET_HAND,
                "batch every person: a body session and a hand session");
    OPB_REQUIRE(bs->net->ctx == hs->net->ctx, "batch every person: both networks must live on the same context");
    OPB_REQUIRE(n >= 1 && n <= 64, "1..64 frames per batch");
    OPB_REQUIRE(H >= 1 && W >= 1, "empty frame");
    OPB_REQUIRE(g_scale > 0, "scale must be positive");
    OPB_REQUIRE(boxsize >= 8 && boxsize % 8 == 0, "boxsize must be a positive multiple of 8 (srcmx/Batch_model.py:377)");
    OPB_CUDA(cudaSetDevice(bs->net->ctx->device));
    cudaStream_t st = bs->stream;
    // the records, the crop tables and the hand plan may still serve the previous batch of this pair, or work of the
    // hand session's own stream
    OPB_CUDA(cudaStreamSynchronize(st));
    OPB_CUDA(cudaStreamSynchronize(hs->stream));
    ensure_every_buffers(bs, 0);
    track_with_tables(hs, boxsize, std::min(H, W));                 // crop tables of every side up to min(H, W)
    FramePlan* fp = get_plan(bs, n, H, W, &g_scale, 1, 2);          // Batch_body on uint8 frames
    ensure_host(bs, n, 0);
    bs->active = fp;
    bs->n_frames = n;
    bs->pose_hand = hs;
    bs->batch_pose_box = boxsize;
    bs->every_batch = true;
    bs->every_persons = -1;
    bs->every_linked = false;
    const double one = 1.0;
    FramePlan* hp = get_plan(hs, kBatchEveryChunk, boxsize, boxsize, &one, 1, 2);   // uint8 Batch_hand on one chunk
    hs->active = hp;
    hs->hand_crops = kBatchEveryChunk;
    hs->hand_ragged = false;
    bs->prof.reset();
    bs->prof.mark(st, "start");
    upload_image(bs, fp, frames, where, (size_t)n * H * W * 3);
    bs->prof.mark(st, "h2d");
    const uint64_t gen = gen_key({bs->buffer_gen, bs->every->gen});
    run_or_replay_slot(bs, GraphSlot{fp->every_graph, fp->every_gen, fp->every_uses}, gen, [&] {
        run_front_f32(bs, fp, n, H, W);
        body_post_enqueue(bs, fp, n, H, W);
        every_rows_enqueue(bs, fp, n);
    });
    OPB_CUDA(cudaEventRecord(bs->done, st));
    bs->net->ctx->launches += fp->launches_per_frame + 1;
}

// ------------------------------------------------------------------------------------------------
// person tracks (opb_tracker_*): the link launch of track.cu on records in device memory
// ------------------------------------------------------------------------------------------------
// track slots for the live tracks plus every person of the frames to link, scratch for the largest frame and for its
// pairs (at most live tracks x persons).  Grown by doubling; OPB_TEST_SMALL_BUFFERS starts tiny so that tests reach the
// growth path.  Waits for `st` before it frees anything.
static void tracker_reserve(opb_tracker* tr, const int* persons, int n, cudaStream_t st) {
    static const bool tiny = getenv("OPB_TEST_SMALL_BUFFERS") != nullptr;
    long long tracks = tr->live, pairs = 0;
    int pmax = 0;
    for (int f = 0; f < n; ++f) {
        OPB_REQUIRE(persons[f] >= 0, "negative person count");
        pairs = std::max(pairs, tracks * persons[f]);
        tracks += persons[f];
        pmax = std::max(pmax, persons[f]);
    }
    OPB_REQUIRE(tracks < (1LL << 30) && pairs < (1LL << 30), "tracker: too many tracks or pairs");
    auto grown = [&](int have, long long need, int first) {
        long long c = have ? have : (tiny ? 2 : first);
        while (c < need) c *= 2;
        return (int)c;
    };
    if (tracks > tr->cap) {
        const int cap = grown(tr->cap, tracks, 256);
        OPB_CUDA(cudaStreamSynchronize(st));
        opb_tracker fresh;      // only its pool and pointers are used
        for (int b = 0; b < 2; ++b) {
            fresh.rows[b] = fresh.tracks.alloc_t<double>((size_t)cap * 54);
            fresh.tid[b] = fresh.tracks.alloc_t<int>(cap);
            fresh.last[b] = fresh.tracks.alloc_t<int>(cap);
        }
        fresh.track_taken = fresh.tracks.alloc_t<int>(cap);
        if (tr->live) {
            const int c = tr->cur, L = tr->live;
            OPB_CUDA(cudaMemcpyAsync(fresh.rows[0], tr->rows[c], (size_t)L * 54 * sizeof(double), cudaMemcpyDeviceToDevice, st));
            OPB_CUDA(cudaMemcpyAsync(fresh.tid[0], tr->tid[c], (size_t)L * sizeof(int), cudaMemcpyDeviceToDevice, st));
            OPB_CUDA(cudaMemcpyAsync(fresh.last[0], tr->last[c], (size_t)L * sizeof(int), cudaMemcpyDeviceToDevice, st));
            OPB_CUDA(cudaStreamSynchronize(st));
        }
        std::swap(tr->tracks.ptrs, fresh.tracks.ptrs);
        std::swap(tr->tracks.bytes, fresh.tracks.bytes);
        for (int b = 0; b < 2; ++b) {
            tr->rows[b] = fresh.rows[b];
            tr->tid[b] = fresh.tid[b];
            tr->last[b] = fresh.last[b];
        }
        tr->track_taken = fresh.track_taken;
        tr->cap = cap;
        tr->cur = 0;
    }
    if (!tr->state || pmax > tr->person_cap || pairs > tr->pair_cap) {
        const int person_cap = std::max(tr->person_cap, grown(tr->person_cap, pmax, 256));
        const int pair_cap = std::max(tr->pair_cap, grown(tr->pair_cap, pairs, 4096));
        OPB_CUDA(cudaStreamSynchronize(st));
        tr->scratch.release();
        tr->person_cap = person_cap;
        tr->pair_cap = pair_cap;
        tr->match = tr->scratch.alloc_t<int>(person_cap);
        tr->pair_cost = tr->scratch.alloc_t<double>(pair_cap);
        tr->pair_k = tr->scratch.alloc_t<int>(pair_cap);
        tr->pair_p = tr->scratch.alloc_t<int>(pair_cap);
        tr->order = tr->scratch.alloc_t<int>(pair_cap);
        tr->state = tr->scratch.alloc_t<int>(5);
        if (!tr->state_host) OPB_CUDA(cudaMallocHost((void**)&tr->state_host, 5 * sizeof(int)));
    }
}

// links n frames (persons_dev / persons_host: the same counts) of records_dev; ids_dev gets one id per record.  The
// state comes back to the pinned buffer; tracker_finish takes it once the stream has reached it.
static void tracker_link_enqueue(opb_tracker* tr, const double* records_dev, const int* persons_dev, const int* persons_host,
                                 int n, int* ids_dev, cudaStream_t st) {
    tracker_reserve(tr, persons_host, n, st);
    TrackLink a;
    a.records = records_dev;
    a.persons = persons_dev;
    a.n_frames = n;
    a.ids = ids_dev;
    for (int b = 0; b < 2; ++b) {
        a.rows[b] = tr->rows[b];
        a.tid[b] = tr->tid[b];
        a.last[b] = tr->last[b];
    }
    a.cap = tr->cap;
    a.person_cap = tr->person_cap;
    a.pair_cap = tr->pair_cap;
    a.cur = tr->cur;
    a.live = tr->live;
    a.next_id = tr->next_id;
    a.frame = tr->frame;
    a.max_gap = tr->max_gap;
    a.min_joints = tr->min_joints;
    a.max_dist = tr->max_dist;
    a.pair_cost = tr->pair_cost;
    a.pair_k = tr->pair_k;
    a.pair_p = tr->pair_p;
    a.order = tr->order;
    a.track_taken = tr->track_taken;
    a.match = tr->match;
    a.state = tr->state;
    OPB_CUDA(cudaMemsetAsync(tr->state, 0, 5 * sizeof(int), st));
    track_link_launch(a, st);
    OPB_CUDA(cudaMemcpyAsync(tr->state_host, tr->state, 5 * sizeof(int), cudaMemcpyDeviceToHost, st));
    tr->ctx->launches += 1;
}

static void tracker_finish(opb_tracker* tr) {
    const int* s = tr->state_host;
    if (s[4]) throw Error(OPB_ERR_INVALID, "tracker: link buffers too small (internal error)");
    tr->cur = s[0];
    tr->live = s[1];
    tr->next_id = s[2];
    tr->frame = s[3];
}

// Body overflow check (frames that overflowed are grown and redone, then the rows-and-boxes kernel runs again), records
// grown to the person count, the hand chunks -- ceil(V / kEveryChunk) Hand chunks, or for an opb_batch_pose_every batch
// ceil(V / kBatchEveryChunk) Batch_hand chunks -- and one copy of the T records.  persons: n ints.  With a tracker,
// frames 0 .. n_link - 1 are linked after the hand chunks and their ids copied back with the records; a batch whose
// Body / Batch_body raised IndexError is not linked.
static int every_wait(opb_session* bs, int* persons, int* frame_status, opb_tracker* tr = nullptr, int n_link = 0) {
    OPB_REQUIRE(bs->active && bs->every && bs->every_batch && bs->pose_hand, "no every-person batch in flight");
    OPB_CUDA(cudaSetDevice(bs->net->ctx->device));
    cudaStream_t st = bs->stream;
    FramePlan* fp = bs->active;
    const int n = bs->n_frames;
    bool again = false;
    const int rc = pose_batch_status(bs, frame_status, again);
    for (;;) {
        if (again) {
            every_rows_enqueue(bs, fp, n);
            OPB_CUDA(cudaStreamSynchronize(st));
        }
        if (bs->every->counts_host[0] <= bs->every->cap) break;
        ensure_every_buffers(bs, bs->every->counts_host[0]);
        again = true;
    }
    opb_session::EveryBuffers& e = *bs->every;
    const int T = e.counts_host[0], V = e.counts_host[1];
    if (V > 0 && bs->batch_pose_box) {
        opb_session* hs = bs->pose_hand;
        FramePlan* hp = hs->active;
        const int boxsize = bs->batch_pose_box;
        const uint64_t gen = gen_key({bs->buffer_gen, hs->buffer_gen, (uint64_t)(uintptr_t)hp, hs->track->gen, e.gen,
                                      (uint64_t)(uintptr_t)fp->d_img, (uint64_t)fp->key.H, (uint64_t)fp->key.W,
                                      (uint64_t)boxsize});
        for (int base = 0; base < V; base += kBatchEveryChunk)
            run_or_replay_slot(bs, GraphSlot{fp->every_hand_graph, fp->every_hand_gen, fp->every_hand_uses}, gen,
                               [&] { batch_every_chunk_enqueue(bs, hs, fp, hp, boxsize); });
        bs->net->ctx->launches += (int64_t)cdiv(V, kBatchEveryChunk) * (3 /* stage, crops, finish */ + hp->launches_per_frame);
    } else if (V > 0) {
        opb_session* hs = bs->pose_hand;
        FramePlan* hp = hs->active;
        const opb_session::Ragged& rg = *hs->ragged;
        const uint64_t gen = gen_key({bs->buffer_gen, hs->buffer_gen, (uint64_t)(uintptr_t)hp, (uint64_t)(uintptr_t)rg.tabs.slab,
                                      (uint64_t)rg.tabs.wmax, e.gen, (uint64_t)(uintptr_t)fp->d_img});
        for (int base = 0; base < V; base += kEveryChunk)
            run_or_replay_slot(bs, GraphSlot{fp->every_hand_graph, fp->every_hand_gen, fp->every_hand_uses}, gen,
                               [&] { every_chunk_enqueue(bs, hs, fp, hp); });
        const int nhs = rg.tabs.n_scales;
        bs->net->ctx->launches += (int64_t)cdiv(V, kEveryChunk) * (1 + nhs + hp->net->kernel_launches + (nhs + 1) + 6 + 1);
    }
    std::unique_lock<std::mutex> lock;
    const bool link = tr && rc == OPB_OK;
    if (link) {
        lock = std::unique_lock<std::mutex>(tr->mu);
        bs->prof.mark(st, "hands");
        if (T > 0) OPB_CUDA(cudaMemsetAsync(e.ids, 0xff, (size_t)T * sizeof(int), st));       // -1: not linked
        tracker_link_enqueue(tr, e.records, e.counts + kEveryFrameCounts, e.counts_host + kEveryFrameCounts, n_link, e.ids, st);
        bs->prof.mark(st, "track_link");
        if (T > 0) OPB_CUDA(cudaMemcpyAsync(e.ids_host, e.ids, (size_t)T * sizeof(int), cudaMemcpyDeviceToHost, st));
    }
    if (T > 0) OPB_CUDA(cudaMemcpyAsync(e.records_host, e.records, (size_t)T * 180 * sizeof(double), cudaMemcpyDeviceToHost, st));
    OPB_CUDA(cudaStreamSynchronize(st));
    if (link) tracker_finish(tr);
    for (int f = 0; f < n; ++f) persons[f] = e.counts_host[kEveryFrameCounts + f];
    bs->every_persons = T;
    bs->every_linked = link;
    return rc;
}

}  // namespace opb

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" {

int opb_abi_version(void) { return OPB_ABI_VERSION; }
const char* opb_last_error(void) { return g_last_error.c_str(); }

int opb_context_create(int device, opb_context** out) {
    return guarded([&] {
        OPB_REQUIRE(out != nullptr, "null out pointer");
        int count = 0;
        if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0)
            throw Error(OPB_ERR_NO_DEVICE, "no CUDA device visible: libopenpose_b200 has no CPU fallback");
        OPB_REQUIRE(device >= 0 && device < count, "device index out of range");
        cudaDeviceProp prop;
        OPB_CUDA(cudaGetDeviceProperties(&prop, device));
        if (prop.major != 10)
            throw Error(OPB_ERR_NO_DEVICE, std::string("device '") + prop.name + "' is sm_" + std::to_string(prop.major) +
                                               std::to_string(prop.minor) + ": this library is built for sm_100a only");
        OPB_CUDA(cudaSetDevice(device));
        auto* c = new opb_context();
        c->device = device;
        c->num_sms = prop.multiProcessorCount;
        OPB_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        *out = c;
    });
}
int opb_context_destroy(opb_context* ctx) {
    return guarded([&] { delete ctx; });
}
int opb_context_synchronize(opb_context* ctx) {
    return guarded([&] {
        OPB_CUDA(cudaSetDevice(ctx->device));
        OPB_CUDA(cudaDeviceSynchronize());
    });
}
int opb_context_launch_count(opb_context* ctx, int64_t* out) {
    return guarded([&] { *out = ctx->launches; });
}

int opb_net_create(opb_context* ctx, int kind, opb_net** out) {
    return guarded([&] {
        OPB_REQUIRE(ctx && out && (kind == OPB_NET_BODY || kind == OPB_NET_HAND), "bad arguments");
        auto* n = new opb_net();
        n->ctx = ctx;
        n->kind = kind;
        *out = n;
    });
}
int opb_net_load_layer(opb_net* net, const char* name, const float* weight, const float* bias, int cout, int cin, int k) {
    return guarded([&] {
        OPB_REQUIRE(net && name && weight && bias && cout > 0 && cin > 0 && k > 0, "bad arguments");
        OPB_REQUIRE(!net->finalized, "net already finalized");
        HostLayer h;
        h.cout = cout; h.cin = cin; h.k = k;
        h.w.assign(weight, weight + (size_t)cout * cin * k * k);
        h.b.assign(bias, bias + cout);
        net->host[name] = std::move(h);
    });
}
int opb_net_finalize(opb_net* net) {
    return guarded([&] { finalize_net(net); });
}
static std::mutex g_lifetime;      // net <-> session reference counts
int opb_net_destroy(opb_net* net) {
    return guarded([&] {
        if (!net) return;
        std::lock_guard<std::mutex> lock(g_lifetime);
        if (net->sessions > 0) {
            net->released = true;          // freed by its last session
            return;
        }
        delete net;
    });
}
int opb_net_layer_count(int kind) {
    if (kind != OPB_NET_BODY && kind != OPB_NET_HAND) return OPB_ERR_INVALID;
    return (int)layer_specs(kind).size();
}
int opb_net_layer_info(int kind, int index, const char** name, int* cout, int* cin, int* k, int* relu) {
    return guarded([&] {
        OPB_REQUIRE(kind == OPB_NET_BODY || kind == OPB_NET_HAND, "bad kind");
        const auto& v = layer_specs(kind);
        OPB_REQUIRE(index >= 0 && index < (int)v.size(), "layer index out of range");
        if (name) *name = v[index].name.c_str();
        if (cout) *cout = v[index].cout;
        if (cin) *cin = v[index].cin;
        if (k) *k = v[index].k;
        if (relu) *relu = v[index].relu ? 1 : 0;
    });
}

int opb_session_create(opb_net* net, opb_session** out) {
    return guarded([&] {
        OPB_REQUIRE(net && out && net->finalized, "net must be finalized first");
        OPB_CUDA(cudaSetDevice(net->ctx->device));
        auto* s = new opb_session();
        s->net = net;
        OPB_CUDA(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
        OPB_CUDA(cudaEventCreateWithFlags(&s->done, cudaEventDisableTiming));
        {
            std::lock_guard<std::mutex> lock(g_lifetime);
            ++net->sessions;
        }
        *out = s;
    });
}
int opb_session_destroy(opb_session* s) {
    return guarded([&] {
        if (!s) return;
        opb_net* net = s->net;
        OPB_CUDA(cudaSetDevice(net->ctx->device));
        cudaStreamSynchronize(s->stream);
        delete s;
        std::lock_guard<std::mutex> lock(g_lifetime);
        if (--net->sessions == 0 && net->released) delete net;
    });
}

int opb_body_submit(opb_session* s, const uint8_t* img, int img_is_device, int H, int W, const double* scales, int ns) {
    return guarded([&] {
        OPB_REQUIRE(s && img && scales, "null argument");
        body_submit(s, img, img_is_device, 1, H, W, scales, ns);
    });
}
int opb_body_submit_batch(opb_session* s, const uint8_t* imgs, int img_is_device, int n_frames, int H, int W,
                          const double* scales, int ns) {
    return guarded([&] {
        OPB_REQUIRE(s && imgs && scales, "null argument");
        body_submit(s, imgs, img_is_device, n_frames, H, W, scales, ns);
    });
}
int opb_body_wait(opb_session* s, int* n_candidate, int* n_subset) {
    int rc = OPB_OK;
    int g = guarded([&] {
        OPB_REQUIRE(s && n_candidate && n_subset, "null argument");
        OPB_REQUIRE(s->n_frames == 1, "a batch is in flight: use opb_body_wait_batch");
        rc = body_wait(s, n_candidate, n_subset, nullptr);
    });
    return g != OPB_OK ? g : rc;
}
int opb_body_wait_batch(opb_session* s, int* n_candidate, int* n_subset, int* frame_status) {
    int rc = OPB_OK;
    int g = guarded([&] {
        OPB_REQUIRE(s && n_candidate && n_subset, "null argument");
        rc = body_wait(s, n_candidate, n_subset, frame_status);
    });
    return g != OPB_OK ? g : rc;
}
int opb_body_fetch(opb_session* s, double* candidate, int cand_rows, double* subset, int subset_rows) {
    return guarded([&] { body_fetch(s, 0, candidate, cand_rows, subset, subset_rows); });
}
int opb_body_fetch_frame(opb_session* s, int frame, double* candidate, int cand_rows, double* subset, int subset_rows) {
    return guarded([&] { body_fetch(s, frame, candidate, cand_rows, subset, subset_rows); });
}

int opb_session_set_profiling(opb_session* s, int on) {
    return guarded([&] {
        OPB_REQUIRE(s != nullptr, "null session");
        s->prof.on = on != 0;
        s->prof.reset();
    });
}
int opb_session_profile_count(opb_session* s) { return s ? (int)s->prof.used : 0; }
int opb_session_profile_get(opb_session* s, int i, const char** name, float* ms_since_prev, double* gflop) {
    return guarded([&] {
        OPB_REQUIRE(s && i >= 0 && i < (int)s->prof.used, "profile index out of range");
        OPB_CUDA(cudaEventSynchronize(s->prof.ev[i]));
        float ms = 0.f;
        if (i > 0) OPB_CUDA(cudaEventElapsedTime(&ms, s->prof.ev[i - 1], s->prof.ev[i]));
        if (name) *name = s->prof.names[i].c_str();
        if (ms_since_prev) *ms_since_prev = ms;
        if (gflop) *gflop = s->prof.gflop[i];
    });
}
/* debug: name of the last profile mark of the in-flight frame that has completed (-1 / "" if none) */
int opb_session_progress(opb_session* s, int* last_done, int* total, const char** name_done, const char** name_next) {
    return guarded([&] {
        OPB_REQUIRE(s && last_done && total, "null argument");
        int done = -1;
        for (int i = 0; i < (int)s->prof.used; ++i) {
            if (cudaEventQuery(s->prof.ev[i]) == cudaSuccess) done = i;
            else break;
        }
        *last_done = done;
        *total = (int)s->prof.used;
        if (name_done) *name_done = done >= 0 ? s->prof.names[done].c_str() : "";
        if (name_next) *name_next = done + 1 < (int)s->prof.used ? s->prof.names[done + 1].c_str() : "";
    });
}
/* timing marks on the session's stream (bench.py): slot 0/1 */
int opb_session_mark(opb_session* s, int slot) {
    return guarded([&] {
        OPB_REQUIRE(s && slot >= 0 && slot < 2, "slot 0 or 1");
        OPB_CUDA(cudaSetDevice(s->net->ctx->device));
        if (!s->marks[slot]) OPB_CUDA(cudaEventCreate(&s->marks[slot]));
        OPB_CUDA(cudaEventRecord(s->marks[slot], s->stream));
    });
}
int opb_session_elapsed(opb_session* a, int slot_a, opb_session* b, int slot_b, float* ms) {
    return guarded([&] {
        OPB_REQUIRE(a && b && ms && a->marks[slot_a] && b->marks[slot_b], "marks not recorded");
        OPB_CUDA(cudaEventSynchronize(a->marks[slot_a]));
        OPB_CUDA(cudaEventSynchronize(b->marks[slot_b]));
        OPB_CUDA(cudaEventElapsedTime(ms, a->marks[slot_a], b->marks[slot_b]));
    });
}

int opb_body_maps(opb_session* s, float* host_heat, float* host_paf) {
    return guarded([&] {
        OPB_REQUIRE(s && s->active && s->net->kind == OPB_NET_BODY, "no finished body frame");
        OPB_CUDA(cudaSetDevice(s->net->ctx->device));
        OPB_CUDA(cudaEventSynchronize(s->done));
        // The frame path never writes the full-resolution maps (peaks.cu / paf.cu evaluate them where needed); they are
        // materialised here, from the net outputs still held by the plan, with the same per-element arithmetic.
        FramePlan* fp = s->active;
        const int n = fp->key.n, H = fp->key.H, W = fp->key.W;
        const size_t px = (size_t)H * W * n;                                                   // all frames of a batch
        bind_maps(s, fp, host_heat != nullptr, host_paf != nullptr, false);
        if (host_heat) {
            run_upsample(fp, false, n, 19, 24, H, W, fp->heat_avg, s->stream);
            OPB_CUDA(cudaMemcpyAsync(host_heat, fp->heat_avg, px * 19 * 4, cudaMemcpyDeviceToHost, s->stream));
        }
        if (host_paf) {
            run_upsample(fp, true, n, 38, 40, H, W, fp->paf_avg, s->stream);
            OPB_CUDA(cudaMemcpyAsync(host_paf, fp->paf_avg, px * 38 * 4, cudaMemcpyDeviceToHost, s->stream));
        }
        OPB_CUDA(cudaStreamSynchronize(s->stream));
    });
}
int opb_hand_maps(opb_session* s, float* host_heat) {
    return guarded([&] {
        OPB_REQUIRE(s && s->active && s->net->kind == OPB_NET_HAND && host_heat, "no finished hand batch");
        OPB_REQUIRE(!s->hand_ragged, "the last hand batch was a list of crops of different sides: its maps have no common shape");
        OPB_CUDA(cudaEventSynchronize(s->done));
        const size_t px = (size_t)s->active->key.H * s->active->key.W;
        OPB_CUDA(cudaMemcpy(host_heat, s->active->heat_avg, px * 22 * 4 * s->active->key.n, cudaMemcpyDeviceToHost));
    });
}

int opb_batch_body_submit(opb_session* s, const float* frames, int where, int n_frames, int H, int W, double g_scale) {
    return guarded([&] {
        OPB_REQUIRE(s && frames, "null argument");
        batch_body_submit(s, frames, false, where, n_frames, H, W, g_scale);
    });
}
int opb_batch_body_submit_u8(opb_session* s, const uint8_t* frames, int where, int n_frames, int H, int W, double g_scale) {
    return guarded([&] {
        OPB_REQUIRE(s && frames, "null argument");
        batch_body_submit(s, frames, true, where, n_frames, H, W, g_scale);
    });
}
int opb_batch_hand_submit(opb_session* s, const float* crops, int where, int n, int H, int W) {
    return guarded([&] {
        OPB_REQUIRE(s && crops, "null argument");
        batch_hand_submit(s, crops, false, where, n, H, W);
    });
}
int opb_batch_hand_submit_u8(opb_session* s, const uint8_t* crops, int where, int n, int H, int W) {
    return guarded([&] {
        OPB_REQUIRE(s && crops, "null argument");
        batch_hand_submit(s, crops, true, where, n, H, W);
    });
}
int opb_batch_maps(opb_session* s, float* host_blurred_heat) {
    return guarded([&] {
        OPB_REQUIRE(s && s->active && s->active->key.mode >= 1 && host_blurred_heat, "no finished batched-estimator call");
        OPB_CUDA(cudaSetDevice(s->net->ctx->device));
        OPB_CUDA(cudaEventSynchronize(s->done));
        FramePlan* fp = s->active;
        const int n = fp->key.n, H = fp->key.H, W = fp->key.W;
        const size_t px = (size_t)H * W * n;
        const int C = s->net->kind == OPB_NET_BODY ? 19 : 22;
        if (s->net->kind == OPB_NET_BODY) {              // body frames: materialised on request only (see opb_body_maps)
            bind_maps(s, fp, true, false, true);
            run_upsample(fp, false, n, 19, 24, H, W, fp->heat_avg, s->stream);
            blur5_planar_launch(fp->heat_avg, fp->blurred, n * 19, H, W, s->stream);
        }
        OPB_CUDA(cudaMemcpyAsync(host_blurred_heat, fp->blurred, px * C * 4, cudaMemcpyDeviceToHost, s->stream));
        OPB_CUDA(cudaStreamSynchronize(s->stream));
    });
}

/* ---- the batched hand job on the device ------------------------------------------------------------------------- */
int opb_hand_track_submit(opb_session* hand_s, const uint8_t* frames_bgr, int where, int n_frames, int height, int width,
                          const double* host_poses, int boxsize) {
    return guarded([&] {
        OPB_REQUIRE(hand_s && frames_bgr && host_poses, "null argument");
        OPB_REQUIRE(where >= 0 && where <= 2, "where: 0 pageable host, 1 device, 2 pinned host");
        hand_track_submit(hand_s, frames_bgr, where, n_frames, height, width, host_poses, boxsize);
    });
}
int opb_hand_track_wait(opb_session* hand_s, double* hand_mats) {
    return guarded([&] {
        OPB_REQUIRE(hand_s && hand_mats && hand_s->track && hand_s->track->n > 0, "no hand-track batch in flight");
        OPB_CUDA(cudaEventSynchronize(hand_s->done));
        memcpy(hand_mats, hand_s->track->mats_host, (size_t)hand_s->track->n * 126 * sizeof(double));
    });
}
int opb_hand_track_crops(opb_session* hand_s, uint8_t* host_crops) {
    return guarded([&] {
        OPB_REQUIRE(hand_s && host_crops && hand_s->track && hand_s->track->plan && hand_s->active == hand_s->track->plan,
                    "the session's last batch was not a hand-track batch");
        OPB_CUDA(cudaSetDevice(hand_s->net->ctx->device));
        OPB_CUDA(cudaEventSynchronize(hand_s->done));
        const FramePlan* fp = hand_s->track->plan;
        OPB_CUDA(cudaMemcpy(host_crops, fp->d_img, (size_t)fp->key.n * fp->key.H * fp->key.W * 3, cudaMemcpyDeviceToHost));
    });
}
int opb_hand_track_boxes(const double* pose54, int height, int width, int* boxes8) {
    return guarded([&] {
        OPB_REQUIRE(pose54 && boxes8 && height >= 1 && width >= 1, "opb_hand_track_boxes: bad argument");
        HandBox hb[2];
        hand_track_boxes_host(pose54, height, width, hb);
        for (int k = 0; k < 2; ++k) {
            boxes8[k * 4 + 0] = hb[k].x;
            boxes8[k * 4 + 1] = hb[k].y;
            boxes8[k * 4 + 2] = hb[k].w;
            boxes8[k * 4 + 3] = hb[k].valid;
        }
    });
}
int opb_debug_hand_track_taps(int side, int boxsize, int* first, float* coef4) {
    return guarded([&] {
        OPB_REQUIRE(first && coef4 && side >= 1 && boxsize >= 1, "opb_debug_hand_track_taps: bad argument");
        const CubicTaps t = hand_track_taps(side, boxsize);
        memcpy(first, t.first.data(), sizeof(int) * boxsize);
        memcpy(coef4, t.coef.data(), sizeof(float) * 4 * boxsize);
    });
}

/* ---- per-frame caller on the device ------------------------------------------------------------------------------ */
int opb_pose_submit_batch(opb_session* body_s, opb_session* hand_s, const uint8_t* imgs, int where, int n_frames, int H,
                          int W, const double* body_scales, int n_body_scales, const double* hand_scales,
                          int n_hand_scales, const int* fixed_boxes) {
    return guarded([&] {
        OPB_REQUIRE(body_s && hand_s && imgs && body_scales && hand_scales, "null argument");
        OPB_REQUIRE(n_hand_scales >= 1 && n_hand_scales <= kMaxScales, "1..8 hand scales");
        pose_submit(body_s, hand_s, imgs, where, n_frames, H, W, body_scales, n_body_scales, hand_scales, n_hand_scales,
                    fixed_boxes);
    });
}
int opb_pose_wait(opb_session* body_s, double* pose_mats, int* frame_status) {
    int rc = OPB_OK;
    int g = guarded([&] {
        OPB_REQUIRE(body_s && pose_mats && body_s->pose && body_s->active && !body_s->batch_pose_box && !body_s->every_batch,
                    "no pose batch in flight");
        // body results first: they report the overflow / IndexError conditions of every frame
        bool grew = false;
        rc = pose_batch_status(body_s, frame_status, grew);
        if (grew) {
            FramePlan* fp = body_s->active;
            opb_session* hs = body_s->pose_hand;
            pose_hand_enqueue(body_s, hs, fp, hs->active, body_s->n_frames, fp->key.H, fp->key.W, body_s->pose_fixed);
            OPB_CUDA(cudaStreamSynchronize(body_s->stream));
        }
        memcpy(pose_mats, body_s->pose->host, (size_t)body_s->n_frames * 180 * sizeof(double));
    });
    return g != OPB_OK ? g : rc;
}

/* ---- the one-pass body + hand job ------------------------------------------------------------------------------- */
int opb_batch_pose_submit(opb_session* body_s, opb_session* hand_s, const uint8_t* frames_bgr, int where, int n_frames,
                          int height, int width, double g_scale, int boxsize) {
    return guarded([&] {
        OPB_REQUIRE(body_s && hand_s && frames_bgr, "null argument");
        OPB_REQUIRE(where >= 0 && where <= 2, "where: 0 pageable host, 1 device, 2 pinned host");
        batch_pose_submit(body_s, hand_s, frames_bgr, where, n_frames, height, width, g_scale, boxsize);
    });
}
int opb_batch_pose_wait(opb_session* body_s, double* motion_mats, double* hand_mats, int* frame_status) {
    int rc = OPB_OK;
    int g = guarded([&] {
        OPB_REQUIRE(body_s && motion_mats && hand_mats && body_s->pose && body_s->active && body_s->batch_pose_box &&
                        !body_s->every_batch, "no batch-pose batch in flight");
        OPB_CUDA(cudaSetDevice(body_s->net->ctx->device));
        bool grew = false;
        rc = pose_batch_status(body_s, frame_status, grew);
        if (grew) {                                   // the hand half again, on the grown frames' new body results
            opb_session* hs = body_s->pose_hand;
            batch_pose_hand_enqueue(body_s, hs, body_s->active, hs->active, body_s->n_frames, body_s->batch_pose_box);
            OPB_CUDA(cudaStreamSynchronize(body_s->stream));
        }
        const double* rec = body_s->pose->host;
        for (int f = 0; f < body_s->n_frames; ++f) {
            memcpy(motion_mats + (size_t)f * 54, rec + (size_t)f * 180, 54 * sizeof(double));
            memcpy(hand_mats + (size_t)f * 126, rec + (size_t)f * 180 + 54, 126 * sizeof(double));
        }
    });
    return g != OPB_OK ? g : rc;
}

/* ---- every person of every frame ------------------------------------------------------------------------------- */
int opb_batch_pose_every_submit(opb_session* body_s, opb_session* hand_s, const uint8_t* frames_bgr, int where,
                                int n_frames, int height, int width, double g_scale, int boxsize) {
    return guarded([&] {
        OPB_REQUIRE(body_s && hand_s && frames_bgr, "null argument");
        OPB_REQUIRE(where >= 0 && where <= 2, "where: 0 pageable host, 1 device, 2 pinned host");
        batch_every_submit(body_s, hand_s, frames_bgr, where, n_frames, height, width, g_scale, boxsize);
    });
}
int opb_pose_every_submit(opb_session* body_s, opb_session* hand_s, const uint8_t* imgs_bgr, int where, int n_frames,
                          int height, int width, const double* body_scales, int n_body_scales, const double* hand_scales,
                          int n_hand_scales) {
    return guarded([&] {
        OPB_REQUIRE(body_s && hand_s && imgs_bgr && body_scales && hand_scales, "null argument");
        OPB_REQUIRE(where >= 0 && where <= 2, "where: 0 pageable host, 1 device, 2 pinned host");
        OPB_REQUIRE(n_hand_scales >= 1 && n_hand_scales <= kMaxScales, "1..8 hand scales");
        every_submit(body_s, hand_s, imgs_bgr, where, n_frames, height, width, body_scales, n_body_scales, hand_scales,
                     n_hand_scales);
    });
}
int opb_pose_every_wait(opb_session* body_s, int* persons, int* frame_status) {
    int rc = OPB_OK;
    int g = guarded([&] {
        OPB_REQUIRE(body_s && persons, "null argument");
        rc = every_wait(body_s, persons, frame_status);
    });
    return g != OPB_OK ? g : rc;
}
int opb_pose_every_fetch(opb_session* body_s, double* records, int rows) {
    return guarded([&] {
        OPB_REQUIRE(body_s && body_s->every && body_s->every_persons >= 0, "no finished every-person batch");
        const int T = body_s->every_persons;
        if (rows < T) throw Error(OPB_ERR_CAPACITY, "records buffer smaller than the result");
        if (T) {
            OPB_REQUIRE(records != nullptr, "null records buffer");
            memcpy(records, body_s->every->records_host, (size_t)T * 180 * sizeof(double));
        }
    });
}
int opb_pose_every_wait_tracked(opb_session* body_s, opb_tracker* tracker, int n_link, int* persons, int* frame_status) {
    int rc = OPB_OK;
    int g = guarded([&] {
        OPB_REQUIRE(body_s && tracker && persons, "null argument");
        OPB_REQUIRE(tracker->ctx == body_s->net->ctx, "tracker and sessions must live on the same context");
        OPB_REQUIRE(n_link >= 0 && n_link <= body_s->n_frames, "n_link: 0..frames of the batch");
        rc = every_wait(body_s, persons, frame_status, tracker, n_link);
    });
    return g != OPB_OK ? g : rc;
}
int opb_pose_every_fetch_ids(opb_session* body_s, int* ids, int rows) {
    return guarded([&] {
        OPB_REQUIRE(body_s && body_s->every && body_s->every_persons >= 0 && body_s->every_linked,
                    "no finished tracked every-person batch");
        const int T = body_s->every_persons;
        if (rows < T) throw Error(OPB_ERR_CAPACITY, "ids buffer smaller than the result");
        if (T) {
            OPB_REQUIRE(ids != nullptr, "null ids buffer");
            memcpy(ids, body_s->every->ids_host, (size_t)T * sizeof(int));
        }
    });
}

/* ---- person tracks ----------------------------------------------------------------------------------------------- */
int opb_tracker_create(opb_context* ctx, int max_gap, double max_dist, int min_joints, opb_tracker** out) {
    return guarded([&] {
        OPB_REQUIRE(ctx && out, "null argument");
        OPB_REQUIRE(max_gap >= 1, "max_gap >= 1");
        OPB_REQUIRE(std::isfinite(max_dist) && max_dist >= 0.0, "max_dist: finite, >= 0");
        OPB_REQUIRE(min_joints >= 1 && min_joints <= 18, "min_joints: 1..18");
        auto* t = new opb_tracker();
        t->ctx = ctx;
        t->max_gap = max_gap;
        t->max_dist = max_dist;
        t->min_joints = min_joints;
        *out = t;
    });
}
int opb_tracker_destroy(opb_tracker* tracker) {
    return guarded([&] {
        if (!tracker) return;
        OPB_CUDA(cudaSetDevice(tracker->ctx->device));
        delete tracker;
    });
}
int opb_tracker_reset(opb_tracker* tracker) {
    return guarded([&] {
        OPB_REQUIRE(tracker, "null argument");
        std::lock_guard<std::mutex> lock(tracker->mu);
        tracker->cur = tracker->live = tracker->next_id = tracker->frame = 0;
    });
}
int opb_tracker_state(opb_tracker* tracker, int* live, int* next_id, int* frame) {
    return guarded([&] {
        OPB_REQUIRE(tracker, "null argument");
        std::lock_guard<std::mutex> lock(tracker->mu);
        if (live) *live = tracker->live;
        if (next_id) *next_id = tracker->next_id;
        if (frame) *frame = tracker->frame;
    });
}
int opb_tracker_link_host(opb_tracker* tracker, const double* records, const int* persons_per_frame, int n_frames, int* ids) {
    return guarded([&] {
        OPB_REQUIRE(tracker && persons_per_frame && n_frames >= 0, "bad arguments");
        long long T = 0;
        for (int f = 0; f < n_frames; ++f) {
            OPB_REQUIRE(persons_per_frame[f] >= 0, "negative person count");
            T += persons_per_frame[f];
        }
        OPB_REQUIRE(T < (1LL << 30), "too many records");
        OPB_REQUIRE(T == 0 || (records && ids), "null argument");
        opb_tracker* tr = tracker;
        OPB_CUDA(cudaSetDevice(tr->ctx->device));
        cudaStream_t st = tr->ctx->stream;
        std::lock_guard<std::mutex> lock(tr->mu);
        if (T > tr->staging_records || n_frames > tr->staging_frames) {
            OPB_CUDA(cudaStreamSynchronize(st));
            tr->staging.release();
            tr->staging_records = (int)std::max<long long>(T, 2 * std::max(tr->staging_records, 0));
            tr->staging_frames = std::max(n_frames, 2 * std::max(tr->staging_frames, 0));
            tr->records = tr->staging.alloc_t<double>((size_t)std::max(tr->staging_records, 1) * 180);
            tr->ids = tr->staging.alloc_t<int>(std::max(tr->staging_records, 1));
            tr->persons = tr->staging.alloc_t<int>(std::max(tr->staging_frames, 1));
        }
        if (T) OPB_CUDA(cudaMemcpyAsync(tr->records, records, (size_t)T * 180 * sizeof(double), cudaMemcpyHostToDevice, st));
        if (n_frames)
            OPB_CUDA(cudaMemcpyAsync(tr->persons, persons_per_frame, (size_t)n_frames * sizeof(int), cudaMemcpyHostToDevice, st));
        tracker_link_enqueue(tr, tr->records, tr->persons, persons_per_frame, n_frames, tr->ids, st);
        if (T) OPB_CUDA(cudaMemcpyAsync(ids, tr->ids, (size_t)T * sizeof(int), cudaMemcpyDeviceToHost, st));
        OPB_CUDA(cudaStreamSynchronize(st));
        tracker_finish(tr);
    });
}

int opb_hand_submit(opb_session* s, const uint8_t* crops, int img_is_device, int n, int H, int W, const double* scales, int ns) {
    return guarded([&] {
        OPB_REQUIRE(s && crops && scales, "null argument");
        hand_submit(s, crops, img_is_device, n, H, W, scales, ns);
    });
}
int opb_hand_submit_ragged(opb_session* s, const uint8_t* packed, const size_t* offsets, int where, int n, const int* sides,
                           const double* scales, int ns) {
    return guarded([&] {
        OPB_REQUIRE(s && packed && offsets && sides && scales, "null argument");
        hand_submit_ragged(s, packed, offsets, where, n, sides, scales, ns);
    });
}
int opb_hand_wait(opb_session* s, double* peaks) {
    return guarded([&] {
        OPB_REQUIRE(s && s->active && peaks, "no frame in flight");
        OPB_CUDA(cudaEventSynchronize(s->done));
        memcpy(peaks, s->hand_host, (size_t)s->hand_crops * 63 * sizeof(double));
    });
}

// ---------------------------------------------------------------------------------------------
// stage-level entry points
// ---------------------------------------------------------------------------------------------
int opb_scale_dims(int H, int W, double scale, int* h, int* w, int* hp, int* wp) {
    return guarded([&] {
        const ScaleDims d = scale_dims(H, W, scale);
        if (h) *h = d.h;
        if (w) *w = d.w;
        if (hp) *hp = d.hp;
        if (wp) *wp = d.wp;
    });
}

int opb_preprocess(opb_context* ctx, const uint8_t* dev_img, int H, int W, double scale, uint8_t* dev_out) {
    return guarded([&] {
        OPB_CUDA(cudaSetDevice(ctx->device));
        const ScaleDims d = scale_dims(H, W, scale);
        DevPool pool;
        TableSlab slab;
        U8Taps t = make_u8_taps(slab, H, W, d);
        t.relocate_to(commit_tables(pool, slab, ctx->stream));
        preprocess_launch(dev_img, H, W, dev_out, d.h, d.w, d.hp, d.wp, t.xf, t.xc, t.yf, t.yc, ctx->stream);
        ctx->launches += 1;
        OPB_CUDA(cudaStreamSynchronize(ctx->stream));
    });
}

int opb_net_forward(opb_session* s, const uint8_t* dev_in, int n, int hp, int wp, float* dev_paf, float* dev_heat) {
    return guarded([&] {
        OPB_REQUIRE(s && dev_in && dev_heat, "null argument");
        OPB_CUDA(cudaSetDevice(s->net->ctx->device));
        std::vector<NetShape> shapes{{n, hp, wp}};
        NetPlan* plan = get_net_plan(s, shapes);
        const size_t px = (size_t)n * (hp / 8) * (wp / 8);
        OPB_CUDA(cudaMemcpyAsync(plan->in_u8[0], dev_in, (size_t)n * hp * wp * 3, cudaMemcpyDeviceToDevice, s->stream));
        plan->run(s->stream);
        if (s->net->kind == OPB_NET_BODY) {
            OPB_REQUIRE(dev_paf != nullptr, "null paf output");
            OPB_CUDA(cudaMemcpyAsync(dev_paf, plan->out_paf[0], px * 40 * 4, cudaMemcpyDeviceToDevice, s->stream));
        }
        OPB_CUDA(cudaMemcpyAsync(dev_heat, plan->out_heat[0], px * 24 * 4, cudaMemcpyDeviceToDevice, s->stream));
        s->net->ctx->launches += plan->kernel_launches;
        OPB_CUDA(cudaStreamSynchronize(s->stream));
    });
}

static NetPlan* debug_plan(opb_session* s) {
    OPB_REQUIRE(s, "null session");
    OPB_REQUIRE(!s->debug_shapes.empty(), "opb_net_debug_plan first");
    OPB_CUDA(cudaSetDevice(s->net->ctx->device));
    return get_net_plan(s, s->debug_shapes);
}
static void fill_debug_step(const NetPlan* plan, int i, opb_debug_step* info) {
    OPB_REQUIRE(i >= 0 && i < (int)plan->steps.size(), "step index out of range");
    if (!info) return;
    const StepInfo& st = plan->step_info[i];
    OPB_REQUIRE((int)st.probs.size() <= OPB_DEBUG_MAX_PROBLEMS, "too many problems in one step");
    memset(info, 0, sizeof(*info));
    info->kind = st.kind;
    info->n_problems = (int)st.probs.size();
    info->block_n = st.block_n;
    info->pool = st.pool;
    info->wide = st.wide;
    info->pair = st.pair;
    info->half_tiles = st.half_tiles;
    info->weights_resident = st.weights_resident;
    snprintf(info->name, sizeof info->name, "%s", plan->step_names[i].c_str());
    auto view = [](const TensorView& t) { return opb_debug_view{t.n, t.h, t.w, t.c, t.cstride, t.coff, t.elem}; };
    for (size_t p = 0; p < st.probs.size(); ++p) {
        const StepProblem& q = st.probs[p];
        snprintf(info->layer[p], sizeof info->layer[p], "%s", q.layer.c_str());
        snprintf(info->layer2[p], sizeof info->layer2[p], "%s", q.layer2.c_str());
        info->scale[p] = q.scale;
        info->in[p] = view(q.in);
        info->out[p] = view(q.out);
    }
}

int opb_net_debug_plan(opb_session* s, int n_scales, const int* shapes, int* n_steps) {
    return guarded([&] {
        OPB_REQUIRE(s && shapes && n_steps && n_scales >= 1 && n_scales <= kMaxScales, "opb_net_debug_plan: bad argument");
        std::vector<NetShape> v;
        for (int i = 0; i < n_scales; ++i) v.push_back({shapes[4 * i], shapes[4 * i + 1], shapes[4 * i + 2], shapes[4 * i + 3]});
        s->debug_shapes = v;
        *n_steps = (int)debug_plan(s)->steps.size();
    });
}
int opb_net_debug_set_input(opb_session* s, int scale, const void* dev_src) {
    return guarded([&] {
        NetPlan* plan = debug_plan(s);
        OPB_REQUIRE(dev_src && scale >= 0 && scale < (int)plan->shapes.size(), "opb_net_debug_set_input: bad argument");
        const NetShape& sh = plan->shapes[scale];
        OPB_CUDA(cudaMemcpyAsync(plan->in_u8[scale], dev_src, (size_t)sh.n * sh.hp * sh.wp * 3 * sh.in_elem,
                                 cudaMemcpyDeviceToDevice, s->stream));
        OPB_CUDA(cudaStreamSynchronize(s->stream));
    });
}
int opb_net_debug_info(opb_session* s, int i, opb_debug_step* info) {
    return guarded([&] { fill_debug_step(debug_plan(s), i, info); });
}
int opb_net_debug_step(opb_session* s, int i, opb_debug_step* info) {
    return guarded([&] {
        NetPlan* plan = debug_plan(s);
        fill_debug_step(plan, i, info);
        plan->steps[i](s->stream);
        s->net->ctx->launches += 1;
        OPB_CUDA(cudaStreamSynchronize(s->stream));
    });
}
int opb_net_debug_read(opb_session* s, int i, int problem, int which, void* dev_dst) {
    return guarded([&] {
        NetPlan* plan = debug_plan(s);
        OPB_REQUIRE(dev_dst && i >= 0 && i < (int)plan->steps.size(), "opb_net_debug_read: bad argument");
        const StepInfo& st = plan->step_info[i];
        OPB_REQUIRE(problem >= 0 && problem < (int)st.probs.size() && (which == 0 || which == 1), "opb_net_debug_read: bad view");
        const TensorView& t = which == 0 ? st.probs[problem].in : st.probs[problem].out;
        OPB_CUDA(cudaMemcpy2DAsync(dev_dst, (size_t)t.c * t.elem, t.ptr(), (size_t)t.cstride * t.elem, (size_t)t.c * t.elem,
                                   t.pixels(), cudaMemcpyDeviceToDevice, s->stream));
        OPB_CUDA(cudaStreamSynchronize(s->stream));
    });
}
int opb_net_debug_run(opb_session* s) {
    return guarded([&] {
        NetPlan* plan = debug_plan(s);
        plan->run(s->stream);
        s->net->ctx->launches += plan->kernel_launches;
        OPB_CUDA(cudaStreamSynchronize(s->stream));
    });
}

// Body (mode 0) / Batch_body (mode 1) post-processing of a frame plan on caller-supplied net outputs
static void check_debug_post(int n_scales, int mode) {
    OPB_REQUIRE(mode == 0 || mode == 1, "mode 0 (Body) or 1 (Batch_body)");
    OPB_REQUIRE(n_scales >= 1 && n_scales <= kMaxScales && (mode == 0 || n_scales == 1),
                "Body takes 1..8 scales, Batch_body one");
}
int opb_body_debug_post_dims(int H, int W, const double* scales, int ns, int mode, int* ho_wo, int* fused) {
    return guarded([&] {
        OPB_REQUIRE(scales && ho_wo && fused, "null argument");
        check_debug_post(ns, mode);
        TableSlab slab;
        std::vector<ScaleDims> dims;
        std::vector<UpTables> tabs;
        for (int i = 0; i < ns; ++i) {
            dims.push_back(plan_dims(H, W, scales[i], mode, true));
            tabs.push_back(make_up_tables(slab, H, W, dims[i], ns));
            ho_wo[2 * i] = dims[i].ho;
            ho_wo[2 * i + 1] = dims[i].wo;
        }
        *fused = plan_fits_fused(tabs, dims, H, W) ? 1 : 0;
    });
}
int opb_body_debug_post_submit(opb_session* s, int n, int H, int W, const double* scales, int ns, int mode,
                               const float* const* heat, const float* const* paf) {
    return guarded([&] {
        OPB_REQUIRE(s && scales && heat && paf, "null argument");
        OPB_REQUIRE(s->net->kind == OPB_NET_BODY, "session was created on a hand network");
        OPB_REQUIRE(n >= 1 && n <= 64, "1..64 frames per batch");
        check_debug_post(ns, mode);
        OPB_CUDA(cudaSetDevice(s->net->ctx->device));
        FramePlan* fp = get_plan(s, n, H, W, scales, ns, mode == 0 ? 0 : 2);
        ensure_host(s, n, 0);
        s->active = fp;
        s->n_frames = n;
        s->prof.reset();
        for (int i = 0; i < ns; ++i) {
            OPB_REQUIRE(heat[i] && paf[i], "null net output");
            const size_t px = (size_t)n * fp->dims[i].ho * fp->dims[i].wo;
            OPB_CUDA(cudaMemcpyAsync(fp->net->out_heat[i], heat[i], px * 24 * sizeof(float), cudaMemcpyHostToDevice, s->stream));
            OPB_CUDA(cudaMemcpyAsync(fp->net->out_paf[i], paf[i], px * 40 * sizeof(float), cudaMemcpyHostToDevice, s->stream));
        }
        body_post_enqueue(s, fp, n, H, W);
        finish_submit(s, fp);
        s->net->ctx->launches -= ns + fp->net->kernel_launches;        // no front end, no CNN
        OPB_CUDA(cudaStreamSynchronize(s->stream));                     // the caller's arrays may be pageable
    });
}
int opb_body_debug_part_begin(opb_session* s, int frame, int* part_begin19) {
    return guarded([&] {
        OPB_REQUIRE(s && part_begin19 && s->active && frame >= 0 && frame < (int)s->results.size(),
                    "no finished frame with this index (opb_body_wait_batch first)");
        memcpy(part_begin19, s->host[frame].counts + 1, 19 * sizeof(int));
    });
}

int opb_upsample_avg(opb_context* ctx, const float* const* dev_maps, const double* scales, int ns, int C, int cstride,
                     int H, int W, float* dev_out) {
    return guarded([&] {
        OPB_REQUIRE(ns >= 1 && ns <= kMaxScales, "1..8 scales");
        OPB_CUDA(cudaSetDevice(ctx->device));
        DevPool pool;
        TableSlab slab;
        std::vector<UpTables> tabs;
        std::vector<ScaleDims> dims;
        size_t scratch = 0;
        for (int i = 0; i < ns; ++i) {
            dims.push_back(scale_dims(H, W, scales[i]));
            tabs.push_back(make_up_tables(slab, H, W, dims[i], ns));
            scratch += (size_t)C * dims[i].ho * W;
        }
        uint8_t* base = commit_tables(pool, slab, ctx->stream);
        UpsampleScale us[kMaxScales];
        for (int i = 0; i < ns; ++i) {
            UpTables& t = tabs[i];
            t.relocate_to(base);
            us[i] = UpsampleScale{dev_maps[i], dims[i].ho, dims[i].wo, cstride, t.xf, t.xw, t.yf, t.yw, t.ybf, t.ybr, t.ybw, t.yb_rs};
        }
        float* tmp = pool.alloc_t<float>(scratch);
        upsample_avg_launch2(us, ns, 1, C, H, W, tmp, dev_out, ctx->stream);
        ctx->launches += ns + 1;
        OPB_CUDA(cudaStreamSynchronize(ctx->stream));
    });
}

// one frame's post-processing buffers for the stage-level entry points
struct StagePost {
    DevPool pool;
    FramePost host;
    FramePost* dev = nullptr;
    int* counters = nullptr;
    void create(int peak_cap, int pair_cap, int conn_cap, int subset_cap, double* ext_candidates, cudaStream_t st) {
        counters = pool.alloc_t<int>(kCounterInts, true);
        alloc_body_post(pool, host, counters, nullptr, peak_cap, pair_cap, conn_cap, subset_cap);
        if (ext_candidates) host.pb.candidates = ext_candidates;
        dev = pool.alloc_t<FramePost>(1);
        OPB_CUDA(cudaMemcpyAsync(dev, &host, sizeof(FramePost), cudaMemcpyHostToDevice, st));
    }
    void clear(cudaStream_t st) { OPB_CUDA(cudaMemsetAsync(counters, 0, kCounterInts * sizeof(int), st)); }
};

static void stage_find_peaks(opb_context* ctx, const float* dev_map, int H, int W, int mode, double thre1,
                             double* dev_candidates, int capacity, int* host_part_begin19, int* n) {
    OPB_REQUIRE(capacity > 0 && dev_candidates && host_part_begin19 && n, "bad arguments");
    OPB_CUDA(cudaSetDevice(ctx->device));
    StagePost sp;
    sp.create(capacity, 1, 1, 1, dev_candidates, ctx->stream);
    MapSource src;
    src.planar = dev_map;
    src.planes_per_frame = 18;
    find_peaks_launch(src, 1, H, W, 18, mode, thre1, sp.dev, nullptr, nullptr, ctx->stream);
    order_peaks_launch(sp.dev, 1, capacity, 18, ctx->stream);
    ctx->launches += 2;
    int appended = 0;
    OPB_CUDA(cudaMemcpyAsync(&appended, sp.host.pb.count, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    OPB_CUDA(cudaMemcpyAsync(host_part_begin19, sp.host.pb.part_begin, 19 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    OPB_CUDA(cudaStreamSynchronize(ctx->stream));
    *n = appended;
    if (appended > capacity) throw Error(OPB_ERR_CAPACITY, "peak buffer too small");
}

int opb_find_peaks(opb_context* ctx, const float* dev_heat, int H, int W, double thre1, double* dev_candidates,
                   int capacity, int* host_part_begin19, int* n) {
    return guarded([&] { stage_find_peaks(ctx, dev_heat, H, W, 0, thre1, dev_candidates, capacity, host_part_begin19, n); });
}

int opb_find_peaks_blurred(opb_context* ctx, const float* dev_blurred, int H, int W, double thre1, double* dev_candidates,
                           int capacity, int* host_part_begin19, int* n) {
    return guarded([&] { stage_find_peaks(ctx, dev_blurred, H, W, 2, thre1, dev_candidates, capacity, host_part_begin19, n); });
}

int opb_smooth_debug(opb_context* ctx, const float* dev_heat, int parts, int H, int W, double* dev_smoothed) {
    return guarded([&] {
        OPB_REQUIRE(dev_heat && dev_smoothed && parts >= 1, "bad arguments");
        OPB_CUDA(cudaSetDevice(ctx->device));
        StagePost sp;
        sp.create(1, 1, 1, 1, nullptr, ctx->stream);
        MapSource src;
        src.planar = dev_heat;
        src.planes_per_frame = parts;
        find_peaks_launch(src, 1, H, W, parts, 0, 1e300, sp.dev, dev_smoothed, nullptr, ctx->stream);
        OPB_CUDA(cudaStreamSynchronize(ctx->stream));
    });
}

int opb_group_limbs(opb_context* ctx, const float* dev_paf, int H, int W, const double* dev_candidates,
                    const int* host_part_begin19, double thre2, double* host_subset, int subset_capacity, int* n_subset,
                    double* host_connections, int conn_capacity, int* host_conn_count19) {
    int rc = OPB_OK;
    int g = guarded([&] {
        OPB_REQUIRE(dev_paf && dev_candidates && host_part_begin19 && host_subset && n_subset, "null argument");
        OPB_CUDA(cudaSetDevice(ctx->device));
        const int total = host_part_begin19[18];
        int max_part = 1;
        for (int p = 0; p < 18; ++p) max_part = std::max(max_part, host_part_begin19[p + 1] - host_part_begin19[p]);
        const int conn_cap = conn_capacity > 0 ? conn_capacity : std::max(1, max_part);
        MapSource src;
        src.planar = dev_paf;
        src.planes_per_frame = 38;
        int status[4], count = 0;
        std::unique_ptr<StagePost> spp;
        // the survivor lists grow on demand, like in the frame path (the reference has no limit)
        int pair_cap = kPairCapacity, rows_cap = std::max(subset_capacity, 1);
        for (;;) {
            spp = std::make_unique<StagePost>();
            spp->create(std::max(total, 1), pair_cap, conn_cap, rows_cap, const_cast<double*>(dev_candidates), ctx->stream);
            OPB_CUDA(cudaMemcpyAsync(spp->host.pb.part_begin, host_part_begin19, 19 * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
            paf_group_launch(src, 1, H, W, spp->dev, thre2, spp->host.lb.subset_capacity, spp->host.lb.pair_capacity,
                             spp->host.lb.max_part, ctx->stream);
            ctx->launches += 4;
            OPB_CUDA(cudaMemcpyAsync(status, spp->host.lb.status, sizeof(status), cudaMemcpyDeviceToHost, ctx->stream));
            OPB_CUDA(cudaMemcpyAsync(&count, spp->host.lb.subset_count, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
            OPB_CUDA(cudaStreamSynchronize(ctx->stream));
            const bool more_pairs = (status[0] & kStPairOverflow) && pair_cap < (1 << 20);
            const bool more_rows = (status[0] & kStSubsetOverflow) && rows_cap < (1 << 16);
            if (!more_pairs && !more_rows) break;
            if (more_pairs) pair_cap *= 4;
            if (more_rows) rows_cap *= 4;      // work rows before pruning; beyond 1024 they live in global memory
        }
        StagePost& sp = *spp;
        if (status[0] & (kStPairOverflow | kStConnOverflow | kStSubsetOverflow))
            throw Error(OPB_ERR_CAPACITY, "limb / person buffers overflowed (status " + std::to_string(status[0]) + ")");
        *n_subset = count;
        if (count > subset_capacity) throw Error(OPB_ERR_CAPACITY, "subset buffer too small");
        if (count) OPB_CUDA(cudaMemcpy(host_subset, sp.host.lb.subset, (size_t)count * 20 * 8, cudaMemcpyDeviceToHost));
        if (host_connections && host_conn_count19) {
            OPB_CUDA(cudaMemcpy(host_conn_count19, sp.host.lb.conn_count, 19 * sizeof(int), cudaMemcpyDeviceToHost));
            OPB_CUDA(cudaMemcpy(host_connections, sp.host.lb.conn, (size_t)19 * conn_cap * 5 * 8, cudaMemcpyDeviceToHost));
        }
        if (status[0] & kStIndexError) {
            set_last_error("list assignment index out of range (src/body.py:173)");
            rc = OPB_ERR_SUBSET_INDEX;
        }
    });
    return g != OPB_OK ? g : rc;
}

int opb_bench_grouping(opb_context* ctx, const float* dev_heat, const float* dev_paf, int H, int W, int iters,
                       float* ms_per_frame, int* n_candidate, int* n_subset) {
    return guarded([&] {
        OPB_REQUIRE(dev_heat && dev_paf && ms_per_frame && iters >= 1, "bad arguments");
        OPB_CUDA(cudaSetDevice(ctx->device));
        StagePost sp;
        sp.create(kPeakCapacity, kPairCapacity, kConnCapacity, kSubsetCapacity, nullptr, ctx->stream);
        MapSource heat, paf;
        heat.planar = dev_heat;
        heat.planes_per_frame = 19;
        paf.planar = dev_paf;
        paf.planes_per_frame = 38;
        cudaEvent_t e0, e1;
        OPB_CUDA(cudaEventCreate(&e0));
        OPB_CUDA(cudaEventCreate(&e1));
        auto once = [&] {
            sp.clear(ctx->stream);
            find_peaks_launch(heat, 1, H, W, 18, 0, 0.1, sp.dev, nullptr, nullptr, ctx->stream);
            order_peaks_launch(sp.dev, 1, sp.host.pb.capacity, 18, ctx->stream);
            paf_group_launch(paf, 1, H, W, sp.dev, 0.05, sp.host.lb.subset_capacity, sp.host.lb.pair_capacity, sp.host.lb.max_part, ctx->stream);
        };
        for (int i = 0; i < 3; ++i) once();
        OPB_CUDA(cudaEventRecord(e0, ctx->stream));
        for (int i = 0; i < iters; ++i) once();
        OPB_CUDA(cudaEventRecord(e1, ctx->stream));
        OPB_CUDA(cudaEventSynchronize(e1));
        float ms = 0.f;
        OPB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        *ms_per_frame = ms / (float)iters;
        ctx->launches += 6 * (iters + 3);
        int pb19[19], ns = 0;
        OPB_CUDA(cudaMemcpy(pb19, sp.host.pb.part_begin, sizeof(pb19), cudaMemcpyDeviceToHost));
        OPB_CUDA(cudaMemcpy(&ns, sp.host.lb.subset_count, sizeof(int), cudaMemcpyDeviceToHost));
        if (n_candidate) *n_candidate = pb19[18];
        if (n_subset) *n_subset = ns;
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
    });
}

/* stage-level: person selection + hand boxes (pose.cu) on host-provided body results */
int opb_pose_select(opb_context* ctx, const double* host_candidates, int n_candidates, const double* host_subset, int n_subset,
                    int H, int W, double* host_pose180, int* host_boxes8) {
    return guarded([&] {
        OPB_REQUIRE(ctx && host_pose180 && host_boxes8 && n_candidates >= 0 && n_subset >= 0, "bad arguments");
        OPB_CUDA(cudaSetDevice(ctx->device));
        StagePost sp;
        sp.create(std::max(n_candidates, 1), 1, 1, std::max(n_subset, 1), nullptr, ctx->stream);
        int pb19[19];
        for (int i = 0; i < 19; ++i) pb19[i] = n_candidates;       // only the total is read
        OPB_CUDA(cudaMemcpyAsync(sp.host.pb.part_begin, pb19, sizeof(pb19), cudaMemcpyHostToDevice, ctx->stream));
        OPB_CUDA(cudaMemcpyAsync(sp.host.lb.subset_count, &n_subset, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
        if (n_candidates)
            OPB_CUDA(cudaMemcpyAsync(sp.host.pb.candidates, host_candidates, (size_t)n_candidates * 32, cudaMemcpyHostToDevice, ctx->stream));
        if (n_subset)
            OPB_CUDA(cudaMemcpyAsync(sp.host.lb.subset, host_subset, (size_t)n_subset * 160, cudaMemcpyHostToDevice, ctx->stream));
        DevPool pool;
        double* pose = pool.alloc_t<double>(180);
        HandBox* boxes = pool.alloc_t<HandBox>(2);
        int* dims = pool.alloc_t<int>(2);
        pose_select_launch(sp.dev, 1, H, W, nullptr, pose, boxes, dims, ctx->stream);
        HandBox hb[2];
        OPB_CUDA(cudaMemcpyAsync(host_pose180, pose, 180 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        OPB_CUDA(cudaMemcpyAsync(hb, boxes, sizeof(hb), cudaMemcpyDeviceToHost, ctx->stream));
        OPB_CUDA(cudaStreamSynchronize(ctx->stream));
        for (int k = 0; k < 2; ++k) {
            host_boxes8[k * 4 + 0] = hb[k].x;
            host_boxes8[k * 4 + 1] = hb[k].y;
            host_boxes8[k * 4 + 2] = hb[k].w;
            host_boxes8[k * 4 + 3] = hb[k].valid;
        }
    });
}

/* stage-level: rows and boxes of every person (pose.cu) on host-provided body results of one frame */
static void every_select(opb_context* ctx, const double* host_candidates, int n_candidates, const double* host_subset,
                         int n_subset, int H, int W, double* host_records, int* host_boxes, bool batched) {
    OPB_REQUIRE(ctx && n_candidates >= 0 && n_subset >= 0, "bad arguments");
    OPB_REQUIRE(n_subset == 0 || (host_candidates && host_subset && host_records && host_boxes), "null argument");
    OPB_CUDA(cudaSetDevice(ctx->device));
    const int cap = std::max(n_subset, 1);
    StagePost sp;
    sp.create(std::max(n_candidates, 1), 1, 1, cap, nullptr, ctx->stream);
    OPB_CUDA(cudaMemcpyAsync(sp.host.lb.subset_count, &n_subset, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    if (n_candidates)
        OPB_CUDA(cudaMemcpyAsync(sp.host.pb.candidates, host_candidates, (size_t)n_candidates * 32, cudaMemcpyHostToDevice, ctx->stream));
    if (n_subset)
        OPB_CUDA(cudaMemcpyAsync(sp.host.lb.subset, host_subset, (size_t)n_subset * 160, cudaMemcpyHostToDevice, ctx->stream));
    DevPool pool;
    double* records = pool.alloc_t<double>((size_t)cap * 180);
    HandBox* list = pool.alloc_t<HandBox>((size_t)cap * 2);
    int* list_rec = pool.alloc_t<int>((size_t)cap * 2);
    int* counts = pool.alloc_t<int>(kEveryCounts);
    every_rows_launch(sp.dev, 1, H, W, cap, records, list, list_rec, counts, batched, ctx->stream);
    ctx->launches += 1;
    std::vector<HandBox> hb((size_t)cap * 2);
    std::vector<int> hr((size_t)cap * 2);
    int hc[kEveryCounts];
    OPB_CUDA(cudaMemcpyAsync(hc, counts, sizeof(hc), cudaMemcpyDeviceToHost, ctx->stream));
    OPB_CUDA(cudaMemcpyAsync(hb.data(), list, hb.size() * sizeof(HandBox), cudaMemcpyDeviceToHost, ctx->stream));
    OPB_CUDA(cudaMemcpyAsync(hr.data(), list_rec, hr.size() * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    if (n_subset)
        OPB_CUDA(cudaMemcpyAsync(host_records, records, (size_t)n_subset * 180 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    OPB_CUDA(cudaStreamSynchronize(ctx->stream));
    OPB_REQUIRE(hc[0] == n_subset && hc[1] <= 2 * n_subset && (!batched || hc[1] == 2 * n_subset),
                "every-person rows: unexpected counts");
    const int fields = batched ? 6 : 5;
    for (int i = 0; i < 2 * n_subset; ++i) {
        int* b = host_boxes + (size_t)i * fields;
        if (i < hc[1]) {
            b[0] = hb[i].x;
            b[1] = hb[i].y;
            b[2] = hb[i].w;
            if (batched) b[3] = hb[i].valid;
            b[fields - 2] = hb[i].left;
            b[fields - 1] = hr[i];
        } else {
            for (int k = 0; k < fields; ++k) b[k] = -1;
        }
    }
}
int opb_pose_every_select(opb_context* ctx, const double* host_candidates, int n_candidates, const double* host_subset,
                          int n_subset, int H, int W, double* host_records, int* host_boxes) {
    return guarded([&] {
        every_select(ctx, host_candidates, n_candidates, host_subset, n_subset, H, W, host_records, host_boxes, false);
    });
}
int opb_batch_pose_every_select(opb_context* ctx, const double* host_candidates, int n_candidates, const double* host_subset,
                                int n_subset, int H, int W, double* host_records, int* host_boxes) {
    return guarded([&] {
        every_select(ctx, host_candidates, n_candidates, host_subset, n_subset, H, W, host_records, host_boxes, true);
    });
}

// The hand post-processing launches of one geometry on caller-supplied planar maps (opb_hand_peaks, opb_hand_debug_post)
static void hand_post(opb_context* ctx, const float* dev_maps, int n_crops, int chan_stride, const int* sides, int H, int W,
                      int mode, int flags, double thre, double* dev_smoothed, int* dev_labels, double* dev_sums,
                      double* host_peaks) {
    OPB_REQUIRE(ctx && dev_maps && host_peaks, "hand post-processing: null argument");
    OPB_REQUIRE(n_crops >= 1 && chan_stride >= 21 && (mode == 0 || mode == 1) && (flags & ~1) == 0,
                "hand post-processing: bad argument");
    OPB_REQUIRE(!sides || mode == 0, "hand post-processing: per-crop sides are a mode-0 geometry");
    OPB_REQUIRE(!dev_smoothed || (mode == 0 && !sides), "hand post-processing: smoothed planes are a mode-0 equal-size output");
    if (sides) {
        H = W = 0;
        for (int c = 0; c < n_crops; ++c) {
            OPB_REQUIRE(sides[c] >= 0, "hand post-processing: negative side");
            H = W = std::max(W, sides[c]);
        }
    }
    OPB_REQUIRE(H >= 1 && W >= 1, "hand post-processing: empty maps");
    OPB_CUDA(cudaSetDevice(ctx->device));
    const size_t planes = (size_t)n_crops * 21 * H * W;
    DevPool pool;
    HandBuffers hb;
    hb.labels = dev_labels ? dev_labels : pool.alloc_t<int>(planes);
    hb.sums = dev_sums ? dev_sums : pool.alloc_t<double>(planes);
    hb.peaks = pool.alloc_t<double>((size_t)n_crops * 63, true);
    hb.exact_all = flags & 1;
    if (mode == 1)
        hand_peaks_blurred_launch(dev_maps, n_crops, chan_stride, H, W, (float)thre, hb, ctx->stream);
    else if (sides)
        hand_peaks_ragged_launch(dev_maps, n_crops, chan_stride, pool.upload(std::vector<int>(sides, sides + n_crops)), W,
                                 thre, hb, ctx->stream);
    else
        hand_peaks_launch2(dev_maps, n_crops, chan_stride, H, W, thre, hb, dev_smoothed, ctx->stream);
    ctx->launches += 6;                  // smooth or mask, runs, merge, compress, flatten, select
    OPB_CUDA(cudaMemcpyAsync(host_peaks, hb.peaks, (size_t)n_crops * 63 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    OPB_CUDA(cudaStreamSynchronize(ctx->stream));
}

int opb_hand_peaks(opb_context* ctx, const float* dev_heat, int H, int W, double thre, double* host_peaks) {
    return guarded([&] { hand_post(ctx, dev_heat, 1, 21, nullptr, H, W, 0, 0, thre, nullptr, nullptr, nullptr, host_peaks); });
}

int opb_hand_debug_post(opb_context* ctx, const float* dev_maps, int n_crops, int chan_stride, const int* sides, int H, int W,
                        int mode, int flags, double* dev_smoothed, int* dev_labels, double* dev_sums, double* host_peaks) {
    return guarded([&] {
        hand_post(ctx, dev_maps, n_crops, chan_stride, sides, H, W, mode, flags, mode == 1 ? (double)0.035f : 0.03,
                  dev_smoothed, dev_labels, dev_sums, host_peaks);
    });
}

int opb_debug_pairwise_sum(const void* values, long long n, int is_f32, double* out) {
    return guarded([&] {
        OPB_REQUIRE(out && n >= 0 && (values || n == 0), "opb_debug_pairwise_sum: bad argument");
        *out = is_f32 ? (double)numpy_sum((const float*)values, n) : numpy_sum((const double*)values, n);
    });
}

int opb_debug_pair_tiles(int n, int h, int w, int n_tiles_n, int small, int* out, int cap, int* written) {
    return guarded([&] {
        OPB_REQUIRE(out && written && n >= 1 && h >= 1 && w >= 1 && n_tiles_n >= 1, "opb_debug_pair_tiles: bad argument");
        const int r = conv_pair_debug_tiles(n, h, w, n_tiles_n, small, out, cap);
        if (r < 0) throw Error(OPB_ERR_CAPACITY, "opb_debug_pair_tiles: output too small");
        *written = r;
    });
}

int opb_debug_resize_taps(int src, int dst, double scale, int* first, float* coef4) {
    return guarded([&] {
        OPB_REQUIRE(first && coef4 && src >= 1 && dst >= 1, "opb_debug_resize_taps: bad argument");
        const CubicTaps t = cubic_taps(src, dst, scale);
        memcpy(first, t.first.data(), sizeof(int) * dst);
        memcpy(coef4, t.coef.data(), sizeof(float) * 4 * dst);
    });
}

int opb_debug_composite_taps(int n_net, int n_resized, int n_orig, int* first, float* w6) {
    return guarded([&] {
        OPB_REQUIRE(first && w6 && n_net >= 1 && n_resized >= 1 && n_resized <= 8 * n_net && n_orig >= 1,
                    "opb_debug_composite_taps: bad argument");
        std::vector<int> f;
        std::vector<float> w;
        composite_taps(n_net, n_resized, n_orig, f, w);
        memcpy(first, f.data(), sizeof(int) * n_orig);
        memcpy(w6, w.data(), sizeof(float) * 6 * n_orig);
    });
}

int opb_debug_resize_dsize(int n, double f) { return resize_dsize(n, f); }

int opb_wide_pool_weights(const float* weight, const float* bias, unsigned short* w_wide, float* b_wide) {
    return guarded([&] {
        OPB_REQUIRE(weight && bias && w_wide && b_wide, "opb_wide_pool_weights: null argument");
        std::vector<__nv_bfloat16> ww;
        std::vector<float> bw;
        wide_pool_weights(weight, bias, ww, bw);
        memcpy(w_wide, ww.data(), ww.size() * sizeof(__nv_bfloat16));
        memcpy(b_wide, bw.data(), bw.size() * sizeof(float));
    });
}

int opb_conv2d(opb_context* ctx, const void* dev_in, int n, int h, int w, int cin, const float* weight, const float* bias,
               int cout, int k, int relu, int pool, int out_fp32, void* dev_out, int impl) {
    return guarded([&] {
        OPB_REQUIRE(cin % 64 == 0, "opb_conv2d: cin must be a multiple of 64");
        OPB_CUDA(cudaSetDevice(ctx->device));
        DevPool dp;
        const int bn = cout <= 64 ? 64 : 128;
        const int cout_pad = (cout + bn - 1) / bn * bn;
        const int cout_store = (cout + 7) / 8 * 8;
        const int taps = k * k;
        const size_t K = (size_t)taps * cin;
        std::vector<__nv_bfloat16> wd((size_t)cout_pad * K, __float2bfloat16_rn(0.f));
        for (int co = 0; co < cout; ++co)
            for (int t = 0; t < taps; ++t)
                for (int c = 0; c < cin; ++c)
                    wd[(size_t)co * K + (size_t)t * cin + c] = __float2bfloat16_rn(weight[((size_t)co * cin + c) * taps + t]);
        std::vector<float> bd(cout_pad, 0.f);
        for (int co = 0; co < cout; ++co) bd[co] = bias[co];
        ConvOp op;
        op.in.base = (void*)dev_in; op.in.n = n; op.in.h = h; op.in.w = w; op.in.c = cin; op.in.cstride = cin; op.in.elem = 2;
        op.out.base = dev_out; op.out.n = n; op.out.h = pool ? h / 2 : h; op.out.w = pool ? w / 2 : w;
        op.out.c = cout_store; op.out.cstride = cout_store; op.out.elem = out_fp32 ? 4 : 2;
        op.w = dp.upload(wd);
        op.bias = dp.upload(bd);
        op.cout_pad = cout_pad; op.cout_store = cout_store; op.ks = k; op.relu = relu != 0; op.pool = pool != 0;
        // impl: 0 = the path the networks use, 1 = scalar cross-check, 2 = per-tap tiles, 3 / 4 = patch MODE 0 / 1,
        // 5 = CTA-pair (cta_group::2) kernel, 6 = the same in the wide-pixel pooled form
        int sel = impl;
        if (impl == 0) sel = (k > 1 && default_conv_impl() >= 0) ? 3 + default_conv_impl() : 2;
        if ((sel == 3 || sel == 4 || sel == 5) && k == 1) sel = 2;
        if (sel == 1) {
            conv_direct_launch(op, ctx->stream);
        } else if (sel == 6) {                       // CTA-pair kernel, wide-pixel pooled form (the networks' conv1_2)
            std::vector<__nv_bfloat16> ww;
            std::vector<float> bw;
            OPB_REQUIRE(cin == 64 && cout == 64 && k == 3, "opb_conv2d: impl 6 is the 64 -> 64 channel 3x3 + pool form");
            wide_pool_weights(weight, bias, ww, bw);
            const ConvOp wide = wide_pool_op(op, dp.upload(ww), dp.upload(bw));
            std::unique_ptr<ConvLaunch> L(conv_pair_plan({wide}, 128, ctx->num_sms));
            L->run(ctx->stream);
        } else if (sel == 2) {
            conv_tc_launch({op}, bn, ctx->stream, ctx->num_sms);
        } else {
            std::unique_ptr<ConvLaunch> L(sel == 5 ? conv_pair_plan({op}, bn, ctx->num_sms)
                                                   : conv_patch_plan({op}, bn, ctx->num_sms, sel - 3));
            L->run(ctx->stream);
        }
        ctx->launches += 1;
        OPB_CUDA(cudaStreamSynchronize(ctx->stream));
    });
}

}  // extern "C"
