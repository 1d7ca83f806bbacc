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
        // util.handDetect on the chosen person (the caller blanks all other rows first, MotionEstimation.py:160-162):
        // left hand from shoulder / elbow / wrist 5, 6, 7, right hand from 2, 3, 4
        for (int k = 0; k < 2; ++k) {
            const int j0 = k == 0 ? 5 : 2;
            const int is = (int)row[j0], ie = (int)row[j0 + 1], iw = (int)row[j0 + 2];
            if (is == -1 || ie == -1 || iw == -1) continue;
            const double x1 = cand[(size_t)is * 4], y1 = cand[(size_t)is * 4 + 1];
            const double x2 = cand[(size_t)ie * 4], y2 = cand[(size_t)ie * 4 + 1];
            const double x3 = cand[(size_t)iw * 4], y3 = cand[(size_t)iw * 4 + 1];
            // an empty box is invalid: the reference's Hand divides by the crop height, it raises there
            hand_detect_box(x1, y1, x2, y2, x3, y3, H, W, hb[k]);
        }
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

// hand key points of slot (frame, k) -> PoseMat rows (MotionEstimation.py:185-194): coordinate 0 means "missing" and
// is not offset; left hands were mirrored: x -> w - x - 1 + x0
__global__ void pose_finish_kernel(const HandBox* __restrict__ boxes, const double* __restrict__ peaks, int n_frames,
                                   double* __restrict__ pose) {
    const int slot = blockIdx.x;
    const int j = threadIdx.x;
    if (j >= 21) return;
    const HandBox b = boxes[slot];
    const int f = slot >> 1;
    double* out = pose + (size_t)f * 180 + (size_t)((b.left ? 18 : 39) + j) * 3;
    if (!b.valid) return;                     // rows stay zero
    const double* p = peaks + ((size_t)slot * 21 + j) * 3;
    double x = p[0], y = p[1];
    if (b.left) x = x == 0 ? x : __dadd_rn(__dadd_rn((double)b.w - x, -1.0), (double)b.x);
    else x = x == 0 ? x : __dadd_rn(x, (double)b.x);
    y = y == 0 ? y : __dadd_rn(y, (double)b.y);
    out[0] = x;
    out[1] = y;
    out[2] = p[2];
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

// Batch_hand key points of slot (frame, k) -> HandMat rows (_box_to_roi, Batch_motion_Estimation.py:41-56): scaled by
// w / boxsize, shifted by the box origin, x un-mirrored for left hands; a coordinate of exactly 0 stays 0.  A slot
// without a box has the box (0, 0, 0): its coordinates become 0 but its scores -- Batch_hand on the grey crop -- stay.
__global__ void hand_track_finish_kernel(const HandBox* __restrict__ boxes, const double* __restrict__ peaks, int boxsize,
                                         double* __restrict__ mats, int frame_stride) {
    const int slot = blockIdx.x;
    const int j = threadIdx.x;
    if (j >= 21) return;
    const HandBox b = boxes[slot];
    const double bx = b.valid ? b.x : 0, by = b.valid ? b.y : 0, bw = b.valid ? b.w : 0;
    const double* p = peaks + ((size_t)slot * 21 + j) * 3;
    const double px = __ddiv_rn(__dmul_rn(p[0], bw), (double)boxsize);
    const double py = __ddiv_rn(__dmul_rn(p[1], bw), (double)boxsize);
    double* out = mats + (size_t)(slot >> 1) * frame_stride + (size_t)((b.left ? 0 : 21) + j) * 3;
    out[0] = px == 0 ? px : (b.left ? __dadd_rn(__dsub_rn(__dsub_rn(bw, px), 1.0), bx) : __dadd_rn(px, bx));
    out[1] = py == 0 ? py : __dadd_rn(py, by);
    out[2] = p[2];
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

}  // namespace

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
