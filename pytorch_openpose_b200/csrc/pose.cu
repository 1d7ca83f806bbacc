// Per-frame caller on the device (srcmx/MotionEstimation.py:126-216, SURVEY.md 8f row N1): from the body results of
// every frame of a batch -- still in device memory -- pick the person, fill the body rows of PoseMat and derive the two
// hand boxes (util.handDetect, src/util.py:133-201); after the hand network, move the hand key points into frame
// coordinates.  PoseMat (60, 3): rows 0-17 body, 18-38 left hand, 39-59 right hand; zeros mean "missing".
// float64 throughout, operation order of the Python code (this file is compiled with --fmad=false).
#include "opb_common.cuh"

namespace opb {
namespace {

// one thread per frame: the work is a few dozen scalar operations
__global__ void pose_select_kernel(const FramePost* __restrict__ frames, int n_frames, int H, int W,
                                   const int* __restrict__ fixed_boxes /* [n][2][3] (x, y, w) left, right or null */,
                                   double* __restrict__ pose, HandBox* __restrict__ boxes, int* __restrict__ dims) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_frames) return;
    const FramePost& fr = frames[f];
    const double* cand = fr.pb.candidates;
    double* pm = pose + (size_t)f * 180;
    for (int i = 0; i < 180; ++i) pm[i] = 0.0;

    // the person (MotionEstimation.py:144-158) and its body rows
    const double* row = select_person_rows(fr, pm);
    HandBox hb[2];
    for (int k = 0; k < 2; ++k) {
        hb[k].frame = f;
        hb[k].x = hb[k].y = hb[k].w = 0;
        hb[k].left = k == 0;
        hb[k].valid = 0;
    }
    if (row) {
        // util.handDetect on the chosen person (the caller blanks all other rows first, MotionEstimation.py:160-162);
        // an empty box is invalid: the reference's Hand divides by the crop height, it raises there
        for (int k = 0; k < 2; ++k) subset_hand_box(cand, row, k, H, W, hb[k]);
    }
    if (fixed_boxes) {                        // benchmarks / tests: random weights find nobody
        for (int k = 0; k < 2; ++k) {
            const int* b = fixed_boxes + ((size_t)f * 2 + k) * 3;
            hb[k].x = b[0];
            hb[k].y = b[1];
            hb[k].w = b[2];
            // a box that is empty or leaves the frame is no box (util.handDetect never produces one)
            hb[k].valid = b[2] > 0 && b[0] >= 0 && b[1] >= 0 && b[0] + b[2] <= W && b[1] + b[2] <= H;
        }
    }
    for (int k = 0; k < 2; ++k) {
        boxes[f * 2 + k] = hb[k];
        dims[f * 2 + k] = hb[k].valid ? hb[k].w : 0;
    }
}

// one hand key point p (x, y, score) of the crop of box b -> its PoseMat row (MotionEstimation.py:185-194): coordinate 0
// means "missing" and is not offset; left hands were mirrored: x -> w - x - 1 + x0
__device__ __forceinline__ void hand_point_to_frame(const HandBox& b, const double* p, double* out) {
    double x = p[0], y = p[1];
    if (b.left) x = x == 0 ? x : __dadd_rn(__dadd_rn((double)b.w - x, -1.0), (double)b.x);
    else x = x == 0 ? x : __dadd_rn(x, (double)b.x);
    y = y == 0 ? y : __dadd_rn(y, (double)b.y);
    out[0] = x;
    out[1] = y;
    out[2] = p[2];
}

// hand key points of slot (frame, k) -> PoseMat rows
__global__ void pose_finish_kernel(const HandBox* __restrict__ boxes, const double* __restrict__ peaks, int n_frames,
                                   double* __restrict__ pose) {
    const int slot = blockIdx.x;
    const int j = threadIdx.x;
    if (j >= 21) return;
    const HandBox b = boxes[slot];
    const int f = slot >> 1;
    double* out = pose + (size_t)f * 180 + (size_t)((b.left ? 18 : 39) + j) * 3;
    if (!b.valid) return;                     // rows stay zero
    hand_point_to_frame(b, peaks + ((size_t)slot * 21 + j) * 3, out);
}

// ---- the batched hand job (srcmx/Batch_motion_Estimation.py:19-63) on saved body poses
// one thread per frame: both hand boxes of poses[f] (n x 18 x 3) in an H x W frame
__global__ void hand_track_boxes_kernel(const double* __restrict__ poses, int n_frames, int H, int W,
                                        HandBox* __restrict__ boxes) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_frames) return;
    HandBox hb[2];
    pose_hand_boxes(poses + (size_t)f * 54, f, H, W, hb);
    boxes[2 * f] = hb[0];
    boxes[2 * f + 1] = hb[1];
}

// one Batch_hand key point p of the crop of box b -> its HandMat row (_box_to_roi, Batch_motion_Estimation.py:41-56):
// scaled by w / boxsize, shifted by the box origin, x un-mirrored for left hands; a coordinate of exactly 0 stays 0.  A
// slot without a box has the box (0, 0, 0): its coordinates become 0 but its score -- Batch_hand on the grey crop --
// stays.
__device__ __forceinline__ void hand_track_point(const HandBox& b, const double* p, int boxsize, double* out) {
    const double bx = b.valid ? b.x : 0, by = b.valid ? b.y : 0, bw = b.valid ? b.w : 0;
    const double px = __ddiv_rn(__dmul_rn(p[0], bw), (double)boxsize);
    const double py = __ddiv_rn(__dmul_rn(p[1], bw), (double)boxsize);
    out[0] = px == 0 ? px : (b.left ? __dadd_rn(__dsub_rn(__dsub_rn(bw, px), 1.0), bx) : __dadd_rn(px, bx));
    out[1] = py == 0 ? py : __dadd_rn(py, by);
    out[2] = p[2];
}

// Batch_hand key points of slot (frame, k) -> HandMat rows
__global__ void hand_track_finish_kernel(const HandBox* __restrict__ boxes, const double* __restrict__ peaks, int boxsize,
                                         double* __restrict__ mats, int frame_stride) {
    const int slot = blockIdx.x;
    const int j = threadIdx.x;
    if (j >= 21) return;
    const HandBox b = boxes[slot];
    hand_track_point(b, peaks + ((size_t)slot * 21 + j) * 3, boxsize,
                     mats + (size_t)(slot >> 1) * frame_stride + (size_t)((b.left ? 0 : 21) + j) * 3);
}

// ---- the one-pass body + hand job: Batch_body_extraction and Batch_hand_extraction (srcmx/Batch_motion_Estimation.py:
// 19-112) on one decode.  One thread per frame of a Batch_body batch: the body rows MotionMat gets (as body_pose on the
// fetched candidates / subset) go into rows 0-17 of records[f] (rows 18-59 zeroed, HandMat lands there later), and the
// hand boxes are derived from exactly those doubles as Batch_hand_extraction derives them from the saved MotionMat
// (HandImageDataset.__getitem__: a joint is missing when x + y + score == 0) -- so both tracks equal the two-pass job's.
__global__ void batch_pose_select_kernel(const FramePost* __restrict__ frames, int n_frames, int H, int W,
                                         double* __restrict__ records, HandBox* __restrict__ boxes) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_frames) return;
    double* rec = records + (size_t)f * 180;
    for (int i = 0; i < 180; ++i) rec[i] = 0.0;
    select_person_rows(frames[f], rec);
    HandBox hb[2];
    pose_hand_boxes(rec, f, H, W, hb);
    boxes[2 * f] = hb[0];
    boxes[2 * f + 1] = hb[1];
}

// ---- every person of every frame (the host loop Body -> util.handDetect -> Hand per box, src/util.py:133-201)
// One block, one thread per frame (n <= 64): person and box counts of every frame, their prefixes, then each thread
// writes its frame's records and boxes.  A frame holds a handful of persons; the loops are a few dozen scalar
// operations per person.
// kBatched: the box rule of the batched estimators (Batch_hand_extraction on the saved MotionMat, as
// batch_pose_select_kernel): both boxes of every person, left then right, from pose_hand_boxes on the record's own body
// rows -- a missing hand is an invalid box that stays in the list (Batch_hand runs on its grey crop), so V = 2T and the
// boxes of record r are entries 2r and 2r + 1.
constexpr int kEveryMaxFrames = 64;
template <bool kBatched>
__global__ void __launch_bounds__(kEveryMaxFrames) every_rows_kernel(const FramePost* __restrict__ frames, int n_frames,
                                                                     int H, int W, int cap, double* __restrict__ records,
                                                                     HandBox* __restrict__ list, int* __restrict__ list_rec,
                                                                     int* __restrict__ counts) {
    __shared__ int s_rec[kEveryMaxFrames + 1], s_box[kEveryMaxFrames + 1];
    const int f = threadIdx.x;
    int persons = 0, boxes = 0;
    if (f < n_frames) {
        const FramePost& fr = frames[f];
        persons = min(*fr.lb.subset_count, fr.lb.subset_capacity);
        if (kBatched) boxes = 2 * persons;
        else for (int p = 0; p < persons; ++p) {
            const double* row = fr.lb.subset + (size_t)p * 20;
            for (int k = 0; k < 2; ++k) {
                const int j0 = k == 0 ? 5 : 2;
                boxes += (int)row[j0] != -1 && (int)row[j0 + 1] != -1 && (int)row[j0 + 2] != -1;
            }
        }
    }
    s_rec[f + 1] = persons;
    s_box[f + 1] = boxes;
    if (f < n_frames) counts[kEveryFrameCounts + f] = persons;
    __syncthreads();
    if (f == 0) {
        s_rec[0] = s_box[0] = 0;
        for (int i = 1; i <= n_frames; ++i) {
            s_rec[i] += s_rec[i - 1];
            s_box[i] += s_box[i - 1];
        }
        counts[0] = s_rec[n_frames];
        counts[1] = s_box[n_frames];
        counts[2] = 0;
    }
    __syncthreads();
    if (f >= n_frames) return;
    const FramePost& fr = frames[f];
    const double* cand = fr.pb.candidates;
    int v = s_box[f];
    for (int p = 0; p < persons; ++p) {
        const int r = s_rec[f] + p;
        const double* row = fr.lb.subset + (size_t)p * 20;
        if (r < cap) {
            double* rec = records + (size_t)r * 180;
            for (int i = 0; i < 180; ++i) rec[i] = 0.0;
            person_rows(cand, row, rec);
            if (kBatched) {                    // v = 2r < 2 cap
                HandBox hb[2];
                pose_hand_boxes(rec, f, H, W, hb);
                for (int k = 0; k < 2; ++k) {
                    list[2 * r + k] = hb[k];
                    list_rec[2 * r + k] = r;
                }
            }
        }
        if (!kBatched) {
            for (int k = 0; k < 2; ++k) {
                HandBox b;
                b.frame = f;
                b.left = k == 0;
                if (!subset_hand_box(cand, row, k, H, W, b)) continue;
                if (v < 2 * cap) {
                    list[v] = b;
                    list_rec[v] = r;
                }
                ++v;
            }
        }
    }
}

// slot i of the chunk <- entry counts[2] + i of the list; past the box count an invalid box (grey crop, no rows)
__global__ void every_stage_kernel(const HandBox* __restrict__ list, const int* __restrict__ list_rec,
                                   const int* __restrict__ counts, int C, HandBox* __restrict__ boxes, int* __restrict__ dims,
                                   int* __restrict__ rec) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= C) return;
    const int v = counts[2] + i;
    HandBox b{};
    int r = -1;
    if (v < counts[1]) {
        b = list[v];
        r = list_rec[v];
    }
    boxes[i] = b;
    dims[i] = b.valid ? b.w : 0;
    rec[i] = r;
}

// the 21 key points of slot `blockIdx.x` into its record (the pose_finish_kernel arithmetic); then the cursor moves on
// to the next chunk -- only this thread touches it, and the next chunk's stage kernel runs after this kernel
__global__ void every_finish_kernel(const HandBox* __restrict__ boxes, const int* __restrict__ rec,
                                    const double* __restrict__ peaks, int C, double* __restrict__ records,
                                    int* __restrict__ counts) {
    const int slot = blockIdx.x;
    const int j = threadIdx.x;
    if (slot == 0 && j == 0) counts[2] += C;
    if (j >= 21) return;
    const HandBox b = boxes[slot];
    if (!b.valid) return;                     // rows stay zero (no box, or a box of width <= 0)
    double* out = records + (size_t)rec[slot] * 180 + (size_t)((b.left ? 18 : 39) + j) * 3;
    hand_point_to_frame(b, peaks + ((size_t)slot * 21 + j) * 3, out);
}

// the batched estimators' chunk finish: slot i's 21 key points into rows 18-38 / 39-59 of record rec[i] with the
// hand_track_finish_kernel arithmetic (_box_to_roi).  Unlike every_finish_kernel, a slot with an invalid box is written
// too -- a missing hand keeps the scores Batch_hand finds on its grey crop, with coordinates 0; slots past V (rec -1)
// are not.  Then the cursor moves on.
__global__ void batch_every_finish_kernel(const HandBox* __restrict__ boxes, const int* __restrict__ rec,
                                          const double* __restrict__ peaks, int C, int boxsize, double* __restrict__ records,
                                          int* __restrict__ counts) {
    const int slot = blockIdx.x;
    const int j = threadIdx.x;
    if (slot == 0 && j == 0) counts[2] += C;
    if (j >= 21) return;
    const int r = rec[slot];
    if (r < 0) return;
    const HandBox b = boxes[slot];
    hand_track_point(b, peaks + ((size_t)slot * 21 + j) * 3, boxsize,
                     records + (size_t)r * 180 + (size_t)((b.left ? 18 : 39) + j) * 3);
}

}  // namespace

void every_rows_launch(const FramePost* frames_dev, int n_frames, int H, int W, int cap, double* records, HandBox* list,
                       int* list_rec, int* counts, bool batched, cudaStream_t stream) {
    OPB_REQUIRE(n_frames >= 1 && n_frames <= kEveryMaxFrames, "1..64 frames per batch");
    if (batched)
        every_rows_kernel<true><<<1, kEveryMaxFrames, 0, stream>>>(frames_dev, n_frames, H, W, cap, records, list, list_rec,
                                                                   counts);
    else
        every_rows_kernel<false><<<1, kEveryMaxFrames, 0, stream>>>(frames_dev, n_frames, H, W, cap, records, list, list_rec,
                                                                    counts);
    OPB_CUDA(cudaGetLastError());
}

void every_stage_launch(const HandBox* list, const int* list_rec, const int* counts, int C, HandBox* boxes, int* dims, int* rec,
                        cudaStream_t stream) {
    every_stage_kernel<<<cdiv(C, 32), 32, 0, stream>>>(list, list_rec, counts, C, boxes, dims, rec);
    OPB_CUDA(cudaGetLastError());
}

void every_finish_launch(const HandBox* boxes, const int* rec, const double* hand_peaks_dev, int C, double* records,
                         int* counts, cudaStream_t stream) {
    every_finish_kernel<<<C, 32, 0, stream>>>(boxes, rec, hand_peaks_dev, C, records, counts);
    OPB_CUDA(cudaGetLastError());
}

void batch_every_finish_launch(const HandBox* boxes, const int* rec, const double* hand_peaks_dev, int C, int boxsize,
                               double* records, int* counts, cudaStream_t stream) {
    batch_every_finish_kernel<<<C, 32, 0, stream>>>(boxes, rec, hand_peaks_dev, C, boxsize, records, counts);
    OPB_CUDA(cudaGetLastError());
}

void hand_track_boxes_host(const double* pose, int H, int W, HandBox* boxes) { pose_hand_boxes(pose, 0, H, W, boxes); }

void hand_track_boxes_launch(const double* poses_dev, int n_frames, int H, int W, HandBox* boxes_dev, cudaStream_t stream) {
    hand_track_boxes_kernel<<<cdiv(n_frames, 64), 64, 0, stream>>>(poses_dev, n_frames, H, W, boxes_dev);
    OPB_CUDA(cudaGetLastError());
}

void hand_track_finish_launch(const HandBox* boxes_dev, const double* hand_peaks_dev, int n_frames, int boxsize,
                              double* mats_dev, int frame_stride, cudaStream_t stream) {
    hand_track_finish_kernel<<<n_frames * 2, 32, 0, stream>>>(boxes_dev, hand_peaks_dev, boxsize, mats_dev, frame_stride);
    OPB_CUDA(cudaGetLastError());
}

void batch_pose_select_launch(const FramePost* frames_dev, int n_frames, int H, int W, double* records_dev,
                              HandBox* boxes_dev, cudaStream_t stream) {
    batch_pose_select_kernel<<<cdiv(n_frames, 64), 64, 0, stream>>>(frames_dev, n_frames, H, W, records_dev, boxes_dev);
    OPB_CUDA(cudaGetLastError());
}

void pose_select_launch(const FramePost* frames_dev, int n_frames, int H, int W, const int* fixed_boxes_dev, double* pose_dev,
                        HandBox* boxes_dev, int* dims_dev, cudaStream_t stream) {
    pose_select_kernel<<<cdiv(n_frames, 64), 64, 0, stream>>>(frames_dev, n_frames, H, W, fixed_boxes_dev, pose_dev, boxes_dev,
                                                             dims_dev);
    OPB_CUDA(cudaGetLastError());
}

void pose_finish_launch(const HandBox* boxes_dev, const double* hand_peaks_dev, int n_frames, double* pose_dev,
                        cudaStream_t stream) {
    pose_finish_kernel<<<n_frames * 2, 32, 0, stream>>>(boxes_dev, hand_peaks_dev, n_frames, pose_dev);
    OPB_CUDA(cudaGetLastError());
}

}  // namespace opb
