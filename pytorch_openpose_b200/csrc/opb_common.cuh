// Shared declarations for the sm_100a OpenPose hot path (internal; the public C ABI is
// include/openpose_b200.h).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>
#include <map>
#include <stdexcept>
#include <memory>
#include <cstring>
#include <cstdlib>

#include "../../include/openpose_b200.h"

namespace opb {

// ---- error plumbing: every C-ABI entry converts exceptions into a code + thread-local message
struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};
void set_last_error(const std::string& m);

#define OPB_CUDA(expr)                                                                          \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess)                                                                  \
            throw opb::Error(OPB_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
    } while (0)

#define OPB_REQUIRE(cond, msg)                                                \
    do {                                                                      \
        if (!(cond)) throw opb::Error(OPB_ERR_INVALID, std::string(msg));     \
    } while (0)

inline int cdiv(int a, int b) { return (a + b - 1) / b; }

// ---- activation tensor view: NHWC, `c` channels starting at element offset `coff` inside rows of
// `cstride` elements (so a conv can read or write a channel slice of a concat buffer in place)
struct TensorView {
    void* base = nullptr;     // start of the underlying buffer (pixel 0, channel 0)
    int n = 1, h = 0, w = 0;  // images, rows, cols
    int c = 0;                // logical channels of this view
    int cstride = 0;          // elements per pixel in the underlying buffer
    int coff = 0;             // first channel of the view
    int elem = 2;             // bytes per element (2 = bf16, 4 = fp32, 1 = u8)
    size_t pixels() const { return (size_t)n * h * w; }
    void* ptr() const { return (char*)base + (size_t)coff * elem; }
};

// ---- tcgen05 implicit-GEMM convolution (conv_tc.cu)
constexpr int kConvMaxProblems = 8;

struct ConvOp {                 // one problem of a grouped launch
    TensorView in;              // bf16 NHWC, c % 64 == 0
    TensorView out;             // bf16 or fp32 NHWC (pooled dims when pool is set)
    const __nv_bfloat16* w;     // [cout_pad][ks*ks*cin] K-major, cin fastest within a tap
    const float* bias;          // [cout_pad]
    int cout_pad = 0;           // multiple of block_n
    int cout_store = 0;         // channels written (multiple of 8, <= cout_pad)
    int ks = 3;                 // 1, 3 or 7 (stride 1, same padding)
    bool relu = true;
    bool pool = false;          // fused 2x2/2 max-pool of the ReLU output
    // "wide pixel" form of a 64 -> 64 channel 3x3 layer followed by the pool (conv1_2; net.cu wide_pool_op): `in` views the
    // image as (h, w/2) pixels of 128 channels (column parity x 64), the 128 output columns are the 64 channels of the even
    // and of the odd column, and the pool is a max over the two column halves and over row pairs.  `kskip` bit
    // (chunk * ks + dx) marks the 64-channel K chunks of a column tap whose weights are all zero: never loaded, never multiplied.
    // `khalf_lo` / `khalf_hi` (same bit index): chunks whose weights are zero for the upper / lower half of the N tile --
    // multiplied as an MMA of half the N extent into that half of the accumulator columns only.
    bool pool_wide = false;
    unsigned kskip = 0, khalf_lo = 0, khalf_hi = 0;
};

void conv_tc_launch(const std::vector<ConvOp>& ops, int block_n, cudaStream_t stream, int num_sms);
// pre-encoded launch (tensor maps + tile list built once per plan, replayed per frame)
struct ConvLaunch {
    int tiles = 0;
    bool half_tiles = false;        // CTA pair: 16 x 8 tiles (plan metadata, for the layer tests)
    bool weights_resident = false;  // CTA pair: bres
    virtual void run(cudaStream_t stream) const = 0;
    virtual ~ConvLaunch() {}
};
ConvLaunch* conv_tc_plan(const std::vector<ConvOp>& ops, int block_n, int num_sms);               // per-tap tiles (any ks)
ConvLaunch* conv_patch_plan(const std::vector<ConvOp>& ops, int block_n, int num_sms, int mode);   // patch-resident (ks 3/7)
ConvLaunch* conv_pair_plan(const std::vector<ConvOp>& ops, int block_n, int num_sms);              // CTA-pair cta_group::2 (ks 3/7)
int conv_pair_debug_tiles(int n, int h, int w, int n_tiles_n, int small, int* out, int cap);        // host only: the kernel's tile list
// fused 1x1 -> ReLU -> 1x1 tail of a refinement stage (conv_tail.cu): in 128 ch -> 128 ch -> cout_store (<= 64) channels
struct TailOp {
    TensorView in, out;
    const __nv_bfloat16 *w1, *w2;   // [128][128] and [64][128], K-major
    const float *b1, *b2;
    int cout_pad2 = 64, cout_store = 0;
    bool relu2 = false;             // ReLU after the second layer (the stage-6 L2 quirk of src/model.py:30-33)
};
bool conv_tail_supported(const std::vector<TailOp>& ops);
ConvLaunch* conv_tail_plan(const std::vector<TailOp>& ops, int num_sms);
// the same with a 512-channel intermediate in four slices (conv5_4 -> conv5_5, conv6_1 -> conv6_2): w1 [512][128], w2 [64][512]
bool conv_tail_wide_supported(const std::vector<TailOp>& ops);
ConvLaunch* conv_tail_wide_plan(const std::vector<TailOp>& ops, int num_sms);
inline void conv_tc_plan_run(const ConvLaunch* L, cudaStream_t stream) { L->run(stream); }
inline void conv_tc_plan_free(ConvLaunch* L) { delete L; }
void tensor_map_encode_bf16(CUtensorMap* tm, void* addr, int rank, const cuuint64_t* dims, const cuuint64_t* strides,
                            const cuuint32_t* box);

// ---- SIMT kernels (conv_simt.cu)
void conv_direct_launch(const ConvOp& op, cudaStream_t stream);                   // debug / cross-check
void conv_first_launch(const TensorView& in_u8, const TensorView& out, const float* w27x64,
                       const float* bias, cudaStream_t stream);                    // conv1_1 (Cin=3) + ReLU
void maxpool2_launch(const TensorView& in, const TensorView& out, cudaStream_t stream);

// Function attributes (dynamic shared memory size) are per device: true the first time `flags` is consulted on the
// current device (one flag array per kernel; contexts on several GPUs may live in one process).
inline bool first_use_on_device(bool (&flags)[64]) {
    int dev = 0;
    cudaGetDevice(&dev);
    dev &= 63;
    if (flags[dev]) return false;
    flags[dev] = true;
    return true;
}

// Programmatic dependent launch (tc_ptx.cuh::pdl_wait): the kernel may start while its predecessor in the stream still
// runs; ONLY for kernels that execute griddepcontrol.wait before they touch the predecessor's output.  OPB_NO_PDL=1
// launches plainly.
template <typename Params>
inline void launch_pdl(void (*kernel)(Params), int grid, int block, size_t smem, cudaStream_t stream, const Params& params) {
    static const bool pdl = getenv("OPB_NO_PDL") == nullptr;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    OPB_CUDA(cudaLaunchKernelEx(&cfg, kernel, params));
}

// ---- pre/post processing (prepost.cu)
void preprocess_launch(const uint8_t* img, int H, int W, uint8_t* out, int h, int w, int hp, int wp,
                       const int* x_first, const short* x_coef, const int* y_first, const short* y_coef,
                       cudaStream_t stream);
void preprocess_launch_batched(const uint8_t* img, int n, int H, int W, uint8_t* out, int h, int w, int hp, int wp,
                               const int* x_first, const short* x_coef, const int* y_first, const short* y_coef,
                               cudaStream_t stream);

// batched estimators (srcmx/Batch_model.py): float frames -> bf16 HWC3 net input; 5x5 blur of planar maps
void preprocess_f32_launch(const void* frames, bool frames_u8_hwc, int n, int H, int W, void* out_bf16, int h, int w,
                           int hp, int wp, const int* x_first, const float* x_w, const int* y_first, const float* y_w,
                           cudaStream_t stream);

constexpr int kUpStrip = 8;          // output rows per register-blocked strip of the y upsample pass (tables + kernel)
struct UpsampleScale {
    const float* src;         // fp32 NHWC net output
    int ho, wo, cstride;      // source dims and per-pixel stride (elements)
    const int* x_first;       // [W]    first source column of the composite footprint
    const float* x_w;         // [W][6] composite weights
    const int* y_first;       // [H]
    const float* y_w;         // [H][6], 1/n_scales folded in
    // optional 16-row strip tables for the register-blocked y pass (null -> generic kernel)
    const int* yb_first = nullptr;     // [ceil(H/16)]
    const int* yb_rows = nullptr;      // [ceil(H/16)]
    const float* yb_w = nullptr;       // [ceil(H/16)][yb_rs][16], 1/n_scales folded in
    int yb_rs = 0;
};
constexpr int kUpTaps = 6;
constexpr int kMaxScales = 8;
void upsample_avg_launch2(const UpsampleScale* scales, int n_scales, int n_img, int C, int H, int W, float* scratch,
                          float* out_planar, cudaStream_t stream);

// ---- composite map: the averaged full-resolution map of src/body.py:54-68 as a FUNCTION of the low-resolution
// net outputs (composite.cuh).  value(ch, y, x) = chain over scales s, taps k of fmaf(yw_s[y][k], t_s(min(yf_s[y]+k,
// ho-1), x), .) with t_s(r, x) = chain over j of fmaf(xw_s[x][j], src_s[r][min(xf_s[x]+j, wo-1)][ch], .) -- the same
// per-element arithmetic as the materialising kernels of prepost.cu, so a value sampled on demand is bit-identical
// to the plane opb_body_maps returns.
struct CompositeScale {
    const float* src;         // fp32 NHWC net output, frame 0
    size_t frame_stride;      // elements between frames
    int ho, wo, cstride;
    const int* xf;            // [W]     first source column
    const float* xw;          // [W][6]
    const int* yf;            // [H]
    const float* yw;          // [H][6]  1/n_scales folded in
    const int* ybf;           // [ceil(H/8)]           strip tables of the register-blocked y pass
    const int* ybr;           // [ceil(H/8)]
    const float* ybw;         // [ceil(H/8)][yb_rs][8]
    int yb_rs;
    // bounds over all output positions (host, float64, rounded outwards): sum of |weights| and range of the sum of
    // weights -- this scale's contribution is <= mid * sum + l1 * halfwidth for inputs in [mid - halfwidth, mid + halfwidth]
    float l1, sum_min, sum_max;
};
struct CompositeMap {
    CompositeScale sc[kMaxScales];
    int n_scales = 0;
    bool fused_ok = false;    // tile footprints fit the fused kernel's shared-memory budget (peaks.cu)
};

// ---- peaks (peaks.cu)
struct PeakBuffers {
    unsigned long long* keys;   // [capacity] unordered (part<<40 | y<<20 | x)
    float* scores;              // [capacity] raw map value, parallel to keys
    int* count;                 // [1] number appended (may exceed capacity -> overflow)
    double* candidates;         // [capacity][4] sorted (x, y, score, id)
    int* part_begin;            // [19] prefix offsets per part (18 parts + total)
    int* part_count;            // [18] scratch of the ordering kernel
    int* ticket;                // [1]  scratch of the ordering kernel (last-block-done counter)
    int capacity;
};

// ---- PAF grouping (paf.cu)
struct LimbBuffers {
    double* cand_score;       // [19][pair_capacity]
    int* cand_ij;             // [19][pair_capacity][2] (i, j)
    int* cand_count;          // [19]
    double* conn;             // [19][conn_capacity][5]  (idA, idB, score, i, j)
    int* conn_count;          // [19]
    double* subset;           // [subset_capacity][20]
    double* rows_global;      // [subset_capacity][kSubsetRowStride] assembly work rows when they do not fit shared memory, else null
    int4* owner_global;       // [max_part] rows holding each candidate (assembly; shared memory is used for small frames)
    int* claim_global;        // [subset_capacity] row claims of the assembly rounds when the rows live in global memory, else null
    int* subset_count;        // [1] rows after pruning
    int* status;              // [4]: bit flags (overflow / IndexError edge), rows before pruning, ...
    int* order;               // [19][pair_capacity] sorted order of the survivors
    int pair_capacity, conn_capacity, subset_capacity, max_part;
};
constexpr int kStPairOverflow = 1, kStConnOverflow = 2, kStSubsetOverflow = 4, kStIndexError = 8;
constexpr int kSubsetRowsShared = 1024;   // assembly rows kept in shared memory up to this many
constexpr int kSubsetRowStride = 21;      // doubles between work rows (20 used)

// everything the post-processing kernels need for ONE frame of a batch; the kernels take a device array of these
// and pick theirs by block index, so a batch is one launch per stage
constexpr int kEagerCand = 2048;      // rows copied to the host before the counts are known
constexpr int kEagerSubset = 128;
struct FrameResults {                // device mirror of the pinned host block, one per frame
    int counts[32];                  // [0] peaks appended, [1..19] part_begin, [20] subset rows, [21..24] status
    double cand[kEagerCand * 4];
    double subset[kEagerSubset * 20];
};
struct FramePost {
    PeakBuffers pb;
    LimbBuffers lb;
    FrameResults* result;     // may be null (stage-level entry points)
};

// where the heat / PAF values come from: materialised planes, or the composite map evaluated on the fly
struct MapSource {
    const float* planar = nullptr;    // (frames * planes_per_frame, H, W) fp32 or null
    int planes_per_frame = 0;
    int frame_base = 0;               // frame index of the first FramePost of the launch (partial re-runs of a batch)
    CompositeMap comp;                // used when planar == null
};

// peak finding over `parts` maps of every frame.  mode 0: sigma-3 Gaussian in scipy's float64 arithmetic, peaks
// scored with the raw value (src/body.py:70-94); mode 1: 5x5 blur in float32, fixed tap order, peaks found and
// scored on the blurred value (srcmx/utilmx.py:230-263); mode 2: mode 1 on a plane that already holds the blurred map.
// Ordered candidates + part_begin are written by
// order_peaks_launch.
// tile_mask_scratch: device words, find_peaks_mask_words(n_frames, H, W) of them (composite sources only).
void find_peaks_launch(const MapSource& src, int n_frames, int H, int W, int parts, int mode, double thre,
                       const FramePost* frames_dev, double* smoothed_out /* mode 0 debug, single frame */,
                       unsigned* tile_mask_scratch, cudaStream_t stream);
size_t find_peaks_mask_words(int n_frames, int H, int W);
// do all tile footprints of a composite map fit the fused kernel's shared-memory budget? (host tables per scale)
bool composite_fits_fused(const std::vector<std::vector<int>>& xf, const std::vector<std::vector<int>>& ybf,
                          const std::vector<std::vector<int>>& ybr, const std::vector<int>& wo, const std::vector<int>& yb_rs,
                          int H, int W);
void order_peaks_launch(const FramePost* frames_dev, int n_frames, int max_capacity, int parts, cudaStream_t stream);
void blur5_planar_launch(const float* maps_planar, float* out_planar, int n_maps, int H, int W, cudaStream_t stream);

// subset_capacity / pair_capacity / max_part: the largest of the launch's frames (grid and shared-memory sizing)
void paf_group_launch(const MapSource& paf, int n_frames, int H, int W, const FramePost* frames_dev, double thre2,
                      int subset_capacity, int pair_capacity, int max_part, cudaStream_t stream);
// copies counts + the first rows of candidates / subsets of every frame into FramePost::result
void pack_results_launch(const FramePost* frames_dev, int n_frames, cudaStream_t stream);

// ---- hand peaks (hand.cu)
struct HandBuffers {
    int* labels;              // [crops*21][h][w]
    double* sums;             // [crops*21][h][w] per-root sums of raw values; scratch of the exact component sums
    double* peaks;            // [crops*21][3] output; [0] / [1] hold the map's sum of |value| and mask count until select
    bool exact_all = false;   // opb_hand_debug_post flag 1: every component gets numpy's sum (sums plane: that sum at its root)
};
void hand_peaks_launch2(const float* heat_planar, int n_crops, int chan_stride_maps, int h, int w, double thre,
                        HandBuffers hb, double* smoothed_out, cudaStream_t stream);
void hand_peaks_blurred_launch(const float* blurred_planar, int n_crops, int chan_stride_maps, int h, int w, float thre,
                               HandBuffers hb, cudaStream_t stream);

// ---- ragged hand crops: per-slot boxes computed on the device and tap tables for every crop size (prepost.cu, pose.cu)
struct HandBox {
    int frame;                // frame of the batch the crop is taken from
    int x, y, w;              // top-left corner and side length in that frame (util.handDetect, src/util.py:133-201)
    int left;                 // left hand: the crop is mirrored before the network, x un-mirrored afterwards
    int valid;                // 0: no box for this slot (no person, missing joints, empty box)
};
// float64 operations rounded once each, on the device and on the host (the units that include this file and call the
// functions below are built without FMA contraction: --fmad=false on the device, baseline x86-64 on the host)
__host__ __device__ inline double dadd_rn(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
__host__ __device__ inline double dmul_rn(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
// np.sum of a contiguous 1-D array of n values in the array's own type (float64 for Hand's raw maps, float32 for
// Batch_hand's blurred maps): numpy's pairwise summation over all n elements, then added to the reduction's +0.0
// (which turns a sum of -0.0s into +0.0).  Every addition rounds once and there are no products to contract, so the
// host and the device produce the same bits.
__host__ __device__ inline long long pairwise_split(long long n) {
    long long n2 = n / 2;
    return n2 - n2 % 8;
}
template <typename T>
__host__ __device__ inline T pairwise_leaf(const T* a, long long n) {           // n <= 128
    if (n < 8) {
        T r = T(0);
        for (long long i = 0; i < n; ++i) r = r + a[i];
        return r;
    }
    T r[8];
    for (int j = 0; j < 8; ++j) r[j] = a[j];
    long long i = 8;
    for (; i < n - n % 8; i += 8)
        for (int j = 0; j < 8; ++j) r[j] = r[j] + a[i + j];
    T res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; ++i) res = res + a[i];
    return res;
}
// pw(a, n) = n <= 128 ? leaf : pw(a, n2) + pw(a + n2, n - n2), walked without recursion (the device stack stays
// small and fixed): leaves are visited left to right; level k of the current path holds the length of its pending
// right half and, once its left half is done, that half's sum.  A split leaves at most n / 2 + 8 values, so 32 levels
// cover any n below 2^36.
template <typename T>
__host__ __device__ inline T pairwise_block(const T* a, long long n) {
    T left[32];
    long long right[32];
    unsigned has_left = 0;                            // bit k: left[k] holds level k's left-half sum
    int sp = 0;
    long long pos = 0, len = n;
    while (true) {
        while (len > 128) {                           // descend along left halves
            const long long n2 = pairwise_split(len);
            right[sp] = len - n2;
            has_left &= ~(1u << sp);
            ++sp;
            len = n2;
        }
        T val = pairwise_leaf(a + pos, len);
        pos += len;
        while (sp > 0 && (has_left >> (sp - 1) & 1)) {   // both halves done: combine and go up
            --sp;
            val = left[sp] + val;
        }
        if (sp == 0) return val;
        left[sp - 1] = val;                           // left half of level sp - 1 done: its right half is next
        has_left |= 1u << (sp - 1);
        len = right[sp - 1];
    }
}
template <typename T>
__host__ __device__ inline T numpy_sum(const T* a, long long n) {
    return T(0) + pairwise_block(a, n);
}

// util.handDetect (src/util.py:133-201) for one arm of one person: shoulder (x1, y1), elbow (x2, y2), wrist (x3, y3) in
// an H x W image -> square box (x, y, w); valid = w > 0 (the reference's crop of an empty box raises)
__host__ __device__ inline void hand_detect_box(double x1, double y1, double x2, double y2, double x3, double y3, int H, int W,
                                                HandBox& b) {
    double x = dadd_rn(x3, dmul_rn(0.33, x3 - x2));
    double y = dadd_rn(y3, dmul_rn(0.33, y3 - y2));
    const double dwe = sqrt(dadd_rn(dmul_rn(x3 - x2, x3 - x2), dmul_rn(y3 - y2, y3 - y2)));
    const double des = sqrt(dadd_rn(dmul_rn(x2 - x1, x2 - x1), dmul_rn(y2 - y1, y2 - y1)));
    const double m = dmul_rn(0.9, des);
    double width = dmul_rn(1.5, dwe > m ? dwe : m);          // max(a, b): a if a > b ... Python's max keeps the first on ties
    x = dadd_rn(x, -(width / 2));
    y = dadd_rn(y, -(width / 2));
    if (x < 0) x = 0;
    if (y < 0) y = 0;
    double w1 = width, w2 = width;
    if (dadd_rn(x, width) > (double)W) w1 = (double)W - x;
    if (dadd_rn(y, width) > (double)H) w2 = (double)H - y;
    width = w2 < w1 ? w2 : w1;                                 // min(width1, width2)
    b.x = (int)x;
    b.y = (int)y;
    b.w = (int)width;
    b.valid = b.w > 0;
}
// HandImageDataset.__getitem__ (srcmx/Batch_model.py:68-104) on a saved (18, 3) pose: joint i is missing when Python's
// sum(pose[i, :]) -- 0 + x + y + score -- is 0; boxes[0] = left hand (joints 5, 6, 7), boxes[1] = right hand (2, 3, 4).
// A hand with a missing joint gets the box (0, 0, 0), invalid.
__host__ __device__ inline void pose_hand_boxes(const double* pose, int frame, int H, int W, HandBox* boxes) {
    for (int k = 0; k < 2; ++k) {
        HandBox& b = boxes[k];
        b.frame = frame;
        b.x = b.y = b.w = 0;
        b.left = k == 0;
        b.valid = 0;
        const int j0 = k == 0 ? 5 : 2;
        bool present = true;
        for (int j = j0; j < j0 + 3; ++j)
            present = present && dadd_rn(dadd_rn(dadd_rn(0.0, pose[j * 3]), pose[j * 3 + 1]), pose[j * 3 + 2]) != 0.0;
        if (present)
            hand_detect_box(pose[j0 * 3], pose[j0 * 3 + 1], pose[(j0 + 1) * 3], pose[(j0 + 1) * 3 + 1], pose[(j0 + 2) * 3],
                            pose[(j0 + 2) * 3 + 1], H, W, b);
    }
}
// the 18 body rows (x, y, score) of one subset row into body54: candidate[subset[k]][:3]; rows of missing joints (-1)
// are left as they are (the callers zero them first)
__device__ inline void person_rows(const double* cand, const double* row, double* body54) {
    for (int k = 0; k < 18; ++k) {
        const int idx = (int)row[k];
        if (idx != -1) {
            body54[k * 3 + 0] = cand[(size_t)idx * 4 + 0];
            body54[k * 3 + 1] = cand[(size_t)idx * 4 + 1];
            body54[k * 3 + 2] = cand[(size_t)idx * 4 + 2];
        }
    }
}
// util.handDetect (src/util.py:133-201) on one subset row: hand k (0 left: shoulder / elbow / wrist 5, 6, 7; 1 right:
// 2, 3, 4).  Returns false, leaving b untouched, when one of the three joints is missing -- handDetect returns no box
// then; otherwise fills x, y, w and valid (b.valid = w > 0: the reference's Hand raises on an empty crop).
__device__ inline bool subset_hand_box(const double* cand, const double* row, int k, int H, int W, HandBox& b) {
    const int j0 = k == 0 ? 5 : 2;
    const int is = (int)row[j0], ie = (int)row[j0 + 1], iw = (int)row[j0 + 2];
    if (is == -1 || ie == -1 || iw == -1) return false;
    const double x1 = cand[(size_t)is * 4], y1 = cand[(size_t)is * 4 + 1];
    const double x2 = cand[(size_t)ie * 4], y2 = cand[(size_t)ie * 4 + 1];
    const double x3 = cand[(size_t)iw * 4], y3 = cand[(size_t)iw * 4 + 1];
    hand_detect_box(x1, y1, x2, y2, x3, y3, H, W, b);
    return true;
}
// the person with the largest left-shoulder x among the body results of one frame (srcmx/MotionEstimation.py:141-158,
// srcmx/Batch_motion_Estimation.py:86-105): a missing shoulder (-1) indexes the LAST candidate, like candidate[-1];
// np.argmax keeps the first maximum.  Writes the person's 18 body rows (x, y, score) into body54 -- rows of missing
// joints are left as they are (the callers zero them first) -- and returns the chosen subset row, or null for nobody.
__device__ inline const double* select_person_rows(const FramePost& fr, double* body54) {
    const double* cand = fr.pb.candidates;
    const int n_cand = fr.pb.part_begin[18];
    const double* subset = fr.lb.subset;
    const int n_sub = *fr.lb.subset_count;
    int chosen = -1;
    double best = 0.0;
    for (int p = 0; p < n_sub; ++p) {
        int idx = (int)subset[(size_t)p * 20 + 5];
        if (idx < 0) idx += n_cand;
        const double x = cand[(size_t)idx * 4];
        if (chosen < 0 || x > best) {
            chosen = p;
            best = x;
        }
    }
    if (chosen < 0) return nullptr;
    const double* row = subset + (size_t)chosen * 20;
    person_rows(cand, row, body54);
    return row;
}

struct RaggedTables {
    const uint8_t* slab;      // all tables
    const unsigned* index;    // [(w * n_scales + s) * 5 + {0: pre first, 1: pre coef, 2: up first, 3: up x weights, 4: up y weights}] byte offsets
    int n_scales, wmax;
};
void preprocess_ragged_launch(const uint8_t* frames, int H, int W, const HandBox* boxes, int n_slots, uint8_t* out, int S,
                              int scale, const RaggedTables& tabs, cudaStream_t stream);
// the same resize with slot i read from its own dense boxes[i].w-square crop at byte offset offsets[i] of `packed`
void preprocess_packed_launch(const uint8_t* packed, const size_t* offsets, const HandBox* boxes, int n_slots, uint8_t* out,
                              int S, int scale, const RaggedTables& tabs, cudaStream_t stream);
void upsample_ragged_launch(const float* const* src, const int* ho, const int* wo, int n_scales, int cstride, int C,
                            const HandBox* boxes, int n_slots, const RaggedTables& tabs, int wmax, float* scratch,
                            float* out_planar, cudaStream_t stream);
void hand_peaks_ragged_launch(const float* heat_planar, int n_crops, int chan_stride_maps, const int* dims_dev, int wmax,
                              double thre, HandBuffers hb, cudaStream_t stream);
// person selection + hand boxes from the body results, and the final PoseMat assembly (pose.cu)
void pose_select_launch(const FramePost* frames_dev, int n_frames, int H, int W, const int* fixed_boxes_dev, double* pose_dev,
                        HandBox* boxes_dev, int* dims_dev, cudaStream_t stream);
void pose_finish_launch(const HandBox* boxes_dev, const double* hand_peaks_dev, int n_frames, double* pose_dev,
                        cudaStream_t stream);
// the batched hand job on saved poses (pose.cu): boxes (2 per frame, left first) and HandMat (n x 42 x 3) assembly
void hand_track_boxes_launch(const double* poses_dev, int n_frames, int H, int W, HandBox* boxes_dev, cudaStream_t stream);
void hand_track_boxes_host(const double* pose, int H, int W, HandBox* boxes);      // the same function on the host
// mats_dev: HandMat of frame f at mats_dev + f * frame_stride (126 for n x 42 x 3, 180 for rows 18-59 of n x 60 x 3)
void hand_track_finish_launch(const HandBox* boxes_dev, const double* hand_peaks_dev, int n_frames, int boxsize,
                              double* mats_dev, int frame_stride, cudaStream_t stream);
// the one-pass body + hand job (pose.cu): from the results of a Batch_body batch, the body rows of a per-frame
// [60][3] record (rows 18-59 zeroed) and both hand boxes derived from those rows as from a saved pose
void batch_pose_select_launch(const FramePost* frames_dev, int n_frames, int H, int W, double* records_dev,
                              HandBox* boxes_dev, cudaStream_t stream);
// every person of every frame (pose.cu).  Rows and boxes: one [60][3] record per subset row (body rows filled, hand
// rows zero), records of frame f from the prefix of the person counts of frames 0..f-1; the boxes util.handDetect
// returns, compacted in its order (frame, person, left before right) into `list` with their record in `list_rec`.
// Records beyond `cap` and boxes beyond 2 * cap are not written.  counts: [0] persons T, [1] boxes V, [2] the chunk
// cursor, reset to 0, [kEveryFrameCounts + f] persons of frame f.  n_frames <= 64.
// batched: the batched estimators' box rule instead (Batch_hand_extraction on each record's body rows, pose_hand_boxes):
// always both boxes of every person, left then right, an invalid one for a missing hand, so V = 2T.
constexpr int kEveryFrameCounts = 4, kEveryCounts = kEveryFrameCounts + 64;
void every_rows_launch(const FramePost* frames_dev, int n_frames, int H, int W, int cap, double* records, HandBox* list,
                       int* list_rec, int* counts, bool batched, cudaStream_t stream);
// one hand chunk: slots [counts[2], counts[2] + C) of the list into boxes / dims / rec (invalid past V); after the hand
// network, the finish scatters each slot's 21 key points into its record and advances counts[2] by C
void every_stage_launch(const HandBox* list, const int* list_rec, const int* counts, int C, HandBox* boxes, int* dims, int* rec,
                        cudaStream_t stream);
void every_finish_launch(const HandBox* boxes, const int* rec, const double* hand_peaks_dev, int C, double* records,
                         int* counts, cudaStream_t stream);
// the batched estimators' finish: Batch_hand key points of a boxsize-square crop -> rows 18-59 of record rec[i]
// (_box_to_roi); a slot with an invalid box keeps its scores with coordinates 0, slots with rec -1 are skipped
void batch_every_finish_launch(const HandBox* boxes, const int* rec, const double* hand_peaks_dev, int C, int boxsize,
                               double* records, int* counts, cudaStream_t stream);

// person tracks across frames (track.cu): links n_frames frames of records (persons[f] records of frame f, one after
// the other, [60][3] each; only rows 0-17 are read) in order, one block.  Track slot k of buffer b: body rows at
// rows[b] + k * 54, id tid[b][k], last matched frame last[b][k]; slots hold ids ascending.  The state in (cur, live,
// next_id, frame) comes as arguments and goes out to state[0..3]; state[4] is set non-zero if a capacity was short
// (cap tracks after adding a frame's persons, person_cap persons per frame, pair_cap eligible pairs per frame).
struct TrackLink {
    const double* records;
    const int* persons;
    int n_frames;
    int* ids;                                 // one per record
    double* rows[2];
    int* tid[2];
    int* last[2];
    int cap, person_cap, pair_cap;
    int cur, live, next_id, frame;
    int max_gap, min_joints;
    double max_dist;
    double* pair_cost;                        // [pair_cap]
    int* pair_k;                              // [pair_cap] track slot
    int* pair_p;                              // [pair_cap] person
    int* order;                               // [pair_cap]
    int* track_taken;                         // [cap]
    int* match;                               // [person_cap] track slot of each person, -1: none
    int* state;                               // [5]
};
void track_link_launch(const TrackLink& a, cudaStream_t stream);

// ---- gaussian taps shared by peaks.cu / hand.cu: scipy.ndimage.gaussian_filter(sigma=3) uses
// radius int(4*3+0.5) = 12 and weights exp(-x^2/18) / sum (src/body.py:75, src/hand.py:62).  The
// constants are the exact float64 bit patterns numpy produces (w[d] = weight at distance d), so the
// device filter can be bit-identical to scipy's.
constexpr int kGaussRadius = 12;
struct GaussTaps {
    double w[kGaussRadius + 1];
};
inline GaussTaps gauss_taps_sigma3() {
    return GaussTaps{{0x1.105a329f98197p-3, 0x1.01a25f86eb137p-3, 0x1.b42a57d56c0bep-4, 0x1.4a614d1afd337p-4,
                      0x1.bfde9c12bec92p-5, 0x1.0fa58939b528fp-5, 0x1.26defcaeb0202p-6, 0x1.1e6bccad344bap-7,
                      0x1.f1e9915139406p-9, 0x1.8345966f69518p-10, 0x1.0d8a5ad43c165p-11, 0x1.4fbe39149e277p-13,
                      0x1.763a210dfb306p-15}};
}

}  // namespace opb
