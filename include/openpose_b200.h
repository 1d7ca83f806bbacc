/*
 * openpose_b200.h -- C ABI of the B200-native OpenPose inference path (libopenpose_b200.so).
 *
 * Drop-in boundary for hitmaxiang/pytorch-openpose (paths relative to the reference checkout):
 *   src/body.py:15-212   class Body   : Body(model_path)(oriImg) -> (candidate, subset)
 *   src/hand.py:16-75    class Hand   : Hand(model_path)(oriImg) -> peaks
 *   src/model.py:25-214  bodypose_model / handpose_model (the two CNNs)
 *   src/util.py:12-40    padRightDownCorner / transfer (checkpoint key mapping)
 * The reference is pure Python over torch/cv2/scipy; a maintainer binds this library with ctypes (see
 * INTEGRATION.md -- pytorch_openpose_b200/_lib.py is exactly that binding).  Plain pointers and sizes
 * only: no torch / numpy / C++ types cross this boundary.
 *
 * Conventions
 *   - every function returns 0 (OPB_OK) or a negative OPB_ERR_* code; opb_last_error() gives the text
 *     for the calling thread.
 *   - "host" pointers are ordinary process memory; "dev" pointers are CUDA device addresses on the
 *     context's device.  All work is issued on the context's stream.
 *   - images are uint8 BGR, HWC, dense (the cv2 layout the reference passes in).
 *   - maps produced on the device are planar fp32: (C, H, W).
 */
#ifndef OPENPOSE_B200_H_
#define OPENPOSE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OPB_ABI_VERSION 1

#define OPB_OK 0
#define OPB_ERR_INVALID (-1)       /* bad argument / shape                                            */
#define OPB_ERR_CUDA (-2)          /* CUDA runtime or driver failure (text in opb_last_error)         */
#define OPB_ERR_MISSING_LAYER (-3) /* checkpoint lacks a layer: the reference's KeyError, util.py:39  */
#define OPB_ERR_CAPACITY (-4)      /* caller buffer too small; required sizes are still returned      */
#define OPB_ERR_SUBSET_INDEX (-5)  /* the reference's IndexError at src/body.py:173 (3rd matching row)*/
#define OPB_ERR_NO_DEVICE (-6)     /* no sm_100 device: this library has no CPU fallback              */

#define OPB_NET_BODY 0
#define OPB_NET_HAND 1

typedef struct opb_context opb_context; /* one per (process, GPU): stream + workspace arena          */
typedef struct opb_net opb_net;         /* weights of one CNN, repacked for the device               */
typedef struct opb_session opb_session; /* per-caller state: plans + buffers for one frame in flight */
typedef struct opb_tracker opb_tracker; /* person tracks of one video (opb_tracker_*)               */

int opb_abi_version(void);
const char* opb_last_error(void);

/* ---- context ------------------------------------------------------------------------------- */
int opb_context_create(int device, opb_context** out);
int opb_context_destroy(opb_context* ctx);
int opb_context_synchronize(opb_context* ctx);
/* number of kernels this library launched on the context since creation (bench.py `gpu_launches`) */
int opb_context_launch_count(opb_context* ctx, int64_t* out);

/* ---- networks: replaces bodypose_model()/handpose_model() + util.transfer + load_state_dict ---- */
/* src/body.py:16-22, src/hand.py:17-23, src/util.py:36-40                                          */
int opb_net_create(opb_context* ctx, int kind, opb_net** out);
/* layer_name is the caffe name without block prefix ("conv1_1", "Mconv7_stage6_L2", ...);
 * weight is OIHW fp32 (cout, cin, k, k), bias fp32 (cout); both host pointers, copied.              */
int opb_net_load_layer(opb_net* net, const char* layer_name, const float* weight, const float* bias,
                       int cout, int cin, int k);
/* Checks every layer of the architecture was provided (else OPB_ERR_MISSING_LAYER naming the first
 * missing one), repacks to bf16 K-major device layout (concat inputs permuted/padded) and uploads.  */
int opb_net_finalize(opb_net* net);
int opb_net_destroy(opb_net* net);
/* number of layers the architecture expects and the i-th layer's name and shape (for host mirrors) */
int opb_net_layer_count(int kind);
int opb_net_layer_info(int kind, int index, const char** name, int* cout, int* cin, int* k, int* relu);

/* ---- sessions ------------------------------------------------------------------------------- */
int opb_session_create(opb_net* net, opb_session** out);
int opb_session_destroy(opb_session* s);

/* Measurement hooks (bench.py).  Profiling records a CUDA event after every stage / convolution launch of the
 * next submitted frame; profile_get(i) returns the name of mark i, the device time since mark i-1 and the
 * algorithmic GFLOP of that launch (0 for non-convolution marks).  mark/elapsed time a region on the session's
 * own stream(s) with CUDA events.                                                                     */
int opb_session_set_profiling(opb_session* s, int on);
int opb_session_profile_count(opb_session* s);
int opb_session_profile_get(opb_session* s, int i, const char** name, float* ms_since_prev, double* gflop);
int opb_session_progress(opb_session* s, int* last_done, int* total, const char** name_done, const char** name_next);
int opb_session_mark(opb_session* s, int slot);
int opb_session_elapsed(opb_session* a, int slot_a, opb_session* b, int slot_b, float* ms);
/* debug: how many launch sequences of the session were captured into a CUDA graph and launched, and how many replayed
 * an already captured graph (the first uses of a job, profiled runs and OPB_NO_GRAPH=1 runs count in neither).      */
int opb_session_graph_stats(opb_session* s, long long* captures, long long* replays);

/* ---- Body.__call__ (src/body.py:24-212) --------------------------------------------------------
 * submit: enqueue the whole frame (H2D of the image when img_is_device == 0, preprocessing at every
 *         scale, CNN, upsample/average, Gaussian+NMS, PAF scoring, matching, assembly, D2H of the
 *         results) on the session's stream without blocking the host.
 * wait  : block until the frame is done; returns the candidate / subset row counts.  A status of
 *         OPB_ERR_SUBSET_INDEX mirrors the reference's IndexError.
 * fetch : copy candidate (n_candidate x 4: x, y, score, id) and subset (n_subset x 20) as float64
 *         row-major into caller memory (src/body.py:160,210-212).                                   */
int opb_body_submit(opb_session* s, const uint8_t* img_bgr, int img_is_device, int height, int width,
                    const double* scale_search, int n_scales);
int opb_body_wait(opb_session* s, int* n_candidate, int* n_subset);
int opb_body_fetch(opb_session* s, double* candidate, int candidate_rows, double* subset, int subset_rows);
/* Batched form (the reference's own throughput path batches frames too: srcmx/Batch_model.py:138-204): n_frames
 * equally sized frames, contiguous (n, H, W, 3), go through every CNN layer in ONE launch per layer; results are
 * per frame.  wait_batch fills n_candidate[n], n_subset[n] and (optionally) frame_status[n] (OPB_OK or
 * OPB_ERR_SUBSET_INDEX per frame) and returns the first non-OK status.                                  */
int opb_body_submit_batch(opb_session* s, const uint8_t* imgs_bgr, int img_is_device, int n_frames, int height,
                          int width, const double* scale_search, int n_scales);
int opb_body_wait_batch(opb_session* s, int* n_candidate, int* n_subset, int* frame_status);
int opb_body_fetch_frame(opb_session* s, int frame, double* candidate, int candidate_rows, double* subset,
                         int subset_rows);

/* Copies the last finished frame's averaged maps to the host: heat (19, H, W) and paf (38, H, W) planar fp32 --
 * the heatmap_avg / paf_avg of src/body.py:33-34,67-68 -- so the reference's own post-processing can be run on
 * the device-produced maps (parity tests).  Either pointer may be NULL.  After a batch the buffers must hold all
 * frames: (n, 19, H, W) and (n, 38, H, W).                                                             */
int opb_body_maps(opb_session* s, float* host_heat, float* host_paf);

/* ---- Hand.__call__ (src/hand.py:25-75) ----------------------------------------------------------
 * n_crops square or rectangular crops of identical size are processed as one batch (the reference
 * calls Hand once per crop; batching is an extension, n_crops == 1 is the drop-in case).
 * peaks: n_crops x 21 x 3 float64 (x, y, score), zeros where nothing exceeds the threshold.          */
int opb_hand_submit(opb_session* s, const uint8_t* crops_bgr, int img_is_device, int n_crops, int height,
                    int width, const double* scale_search, int n_scales);
int opb_hand_wait(opb_session* s, double* peaks);
/* n_crops square crops of any sides as one batch: crop i is the dense sides[i] x sides[i] x 3 uint8 BGR image at
 * bytes [offsets[i], offsets[i + 1]) of `packed` (n_crops + 1 offsets, offsets[0] = 0, crops back to back; `where`
 * as opb_body_submit for the whole packed buffer).  Row i of the peaks equals opb_hand_submit on crop i alone, bit
 * for bit.  The scales must resize every square crop to a net input whose side is a multiple of 8 (the default
 * 0.5, 1, 1.5, 2 do).  Results: opb_hand_wait; opb_hand_maps refuses such a batch (its maps have no common shape). */
int opb_hand_submit_ragged(opb_session* s, const uint8_t* packed, const size_t* offsets, int where, int n_crops,
                           const int* sides, const double* scale_search, int n_scales);
/* heatmap_avg of the last hand batch: (n_crops, 22, h, w) planar fp32 (src/hand.py:33,57).             */
int opb_hand_maps(opb_session* s, float* host_heat);

/* ---- the per-frame caller on the device: MotionData_every_frame(mode='bodyhand') ------------------
 * srcmx/MotionEstimation.py:126-216 for a batch of equally sized frames: body estimation, selection of the
 * person with the largest left-shoulder x (:144-162), util.handDetect (src/util.py:133-201), both hand
 * crops taken -- the left one mirrored -- from the frame that is already on the device, Hand on all 2 * n
 * crops as one ragged batch (every slot keeps its own crop size), key points moved back to frame
 * coordinates (:185-194).  The only result copied to the host is PoseMat: n x 60 x 3 float64 (rows 0-17
 * body, 18-38 left hand, 39-59 right hand; zeros = missing).  hand_s must not be used by other calls
 * while a pose batch is in flight.  fixed_boxes (optional, host, n x 2 x 3 ints: x, y, w of the left and
 * the right hand box; w <= 0 = none) replaces handDetect's boxes (benchmarks with random weights, which
 * find no person).  wait returns the first non-OK frame status like opb_body_wait_batch; an empty hand
 * box (width 0), on which the reference's Hand raises ZeroDivisionError, yields zero rows.            */
int opb_pose_submit_batch(opb_session* body_s, opb_session* hand_s, const uint8_t* imgs_bgr, int where, int n_frames,
                          int height, int width, const double* body_scales, int n_body_scales,
                          const double* hand_scales, int n_hand_scales, const int* fixed_boxes);
int opb_pose_wait(opb_session* body_s, double* pose_mats, int* frame_status);
/* ---- every person of every frame ----------------------------------------------------------------------------------
 * The caller's loop over everyone Body finds, for a batch of equally sized uint8 BGR frames: per frame, one 60 x 3
 * float64 record per subset row, in subset order (rows 0-17 candidate[subset[p][k]][:3], zero where the index is -1),
 * util.handDetect on every subset row (src/util.py:133-201), Hand on every box it returns -- the left crop mirrored --
 * and the key points in frame coordinates in rows 18-38 (left) and 39-59 (right) of the box's person, as
 * srcmx/MotionEstimation.py:185-194 computes them.  A hand with a missing joint gets zero rows and no crop; a box of
 * width <= 0, on which the reference's Hand raises ZeroDivisionError, gives zero rows.  Arguments as
 * opb_pose_submit_batch (1 <= n_frames <= 64, `where`: 0 pageable host, 1 device, 2 pinned host).  The hand crops run
 * in fixed chunks of 8 through one hand plan, so memory does not depend on the number of persons.  hand_s must not be
 * used by other calls while a batch is in flight.
 * wait: runs the hand chunks, fills persons (n ints: records of each frame) and frame_status (optional: OPB_OK or
 * OPB_ERR_SUBSET_INDEX per frame), returns the first non-OK status like opb_body_wait_batch.
 * fetch: the records of the last wait, frame after frame (sum of persons x 60 x 3); rows = capacity of `records` in
 * records.
 * wait, fetch, wait_tracked and fetch_ids below serve both opb_pose_every_submit and opb_batch_pose_every_submit: the
 * wait runs the hand chunks of whichever submit put the batch in flight.                                          */
int opb_pose_every_submit(opb_session* body_s, opb_session* hand_s, const uint8_t* imgs_bgr, int where, int n_frames,
                          int height, int width, const double* body_scales, int n_body_scales,
                          const double* hand_scales, int n_hand_scales);
int opb_pose_every_wait(opb_session* body_s, int* persons, int* frame_status);
int opb_pose_every_fetch(opb_session* body_s, double* records, int rows);
/* ---- person tracks across frames ----------------------------------------------------------------------------------
 * A tracker links the persons of consecutive frames into tracks with the rule of motion.PersonLinker (its docstring is
 * the specification; the ids are bit-identical): presence = score > 0, cost = mean joint distance over the >= min_joints
 * body joints present in both, eligible when <= max_dist, greedy matching on (cost, track id, person), unmatched persons
 * open new tracks (ids 0, 1, ... in creation order, never reused), a track unmatched for more than max_gap frames is
 * dropped.  One tracker follows one video: frames are linked in the order the calls return.  Calls on one tracker are
 * serialised by a mutex and each ends in a stream synchronise, so two session pairs may alternate on it.
 * create: max_gap >= 1, max_dist finite >= 0, 1 <= min_joints <= 18.  reset: forget every track (next frame 0, next
 * id 0).  state: live tracks, next id, frames linked so far (each pointer optional).
 * wait_tracked: opb_pose_every_wait, then frames 0 .. n_link - 1 of the batch (0 <= n_link <= n) linked on the device
 * in the same stream; frames past n_link (a padded batch) do not advance the tracker and get id -1.  A batch with a
 * non-OK status is not linked.  fetch_ids: the ids of the last tracked wait, one per record, in record order.
 * link_host: the same link launch on host records (persons_per_frame[f] records of 60 x 3 doubles for frame f, one
 * frame after the other) -> ids, one per record (parity tests, foreign estimators).                               */
int opb_tracker_create(opb_context* ctx, int max_gap, double max_dist, int min_joints, opb_tracker** out);
int opb_tracker_destroy(opb_tracker* tracker);
int opb_tracker_reset(opb_tracker* tracker);
int opb_tracker_state(opb_tracker* tracker, int* live, int* next_id, int* frame);
int opb_pose_every_wait_tracked(opb_session* body_s, opb_tracker* tracker, int n_link, int* persons, int* frame_status);
int opb_pose_every_fetch_ids(opb_session* body_s, int* ids, int rows);
int opb_tracker_link_host(opb_tracker* tracker, const double* records, const int* persons_per_frame, int n_frames,
                          int* ids);

/* ---- batched estimators: srcmx/Batch_model.py (the reference author's throughput path) ---------- */
/* Batch_body.__call__ (srcmx/Batch_model.py:142-204): `frames` = (n, 3, height, width) float32 planar in
 * [0,1] (torchvision ToTensor), one scale g_scale (the reference uses 0.5, :118) with truncating sizes
 * (:340-345), torch bicubic resizes, zero padding after the -0.5 shift, 5x5 blur of the full-size heat
 * maps (srcmx/utilmx.py:243-263), peaks found and scored on the BLURRED maps (utilmx.py:230-241,
 * Batch_model.py:194), grouping as Body (Batch_model.py:206-338).  `where`: 0 pageable host, 1 device,
 * 2 pinned host.  Results: opb_body_wait_batch / opb_body_fetch_frame.                               */
int opb_batch_body_submit(opb_session* s, const float* frames, int where, int n_frames, int height, int width,
                          double g_scale);
/* Batch_hand.__call__ (srcmx/Batch_model.py:366-406): `crops` = (n, 3, height, width) float32 in [0,1],
 * no resize, x8 bicubic upsampling, 5x5 blur, threshold 0.035 / component sums / maximum all on the
 * blurred maps.  height and width must be multiples of 8.  Results: opb_hand_wait.                  */
int opb_batch_hand_submit(opb_session* s, const float* crops, int where, int n_crops, int height, int width);
/* The same two calls on frames as they come out of the decoder: (n, height, width, 3) uint8; the division by 255
 * of torchvision's ToTensor (srcmx/Batch_model.py:409, :101-102) is applied on the device, bit-identically, so the
 * host neither converts nor uploads float pixels.                                                     */
int opb_batch_body_submit_u8(opb_session* s, const uint8_t* frames_hwc, int where, int n_frames, int height, int width,
                             double g_scale);
int opb_batch_hand_submit_u8(opb_session* s, const uint8_t* crops_hwc, int where, int n_crops, int height, int width);
/* ---- Batch_hand_extraction (srcmx/Batch_motion_Estimation.py:19-63) on the device --------------------------------
 * For n_frames ROI-cropped frames (n, height, width, 3) uint8 and their saved body poses (host, n x 18 x 3 float64, the
 * track Batch_body_extraction writes): both hand boxes of every pose (HandImageDataset.__getitem__,
 * srcmx/Batch_model.py:68-104 -- a joint is missing when x + y + score == 0, util.handDetect on the one person), the
 * crops cv2.resize(crop, (boxsize, boxsize), INTER_CUBIC), the left one mirrored, a uniform 128 image where a hand is
 * missing, Batch_hand on all 2n crops (as opb_batch_hand_submit_u8), and the key points moved back to ROI coordinates
 * (Batch_motion_Estimation.py:41-56).  `where`: 0 pageable host, 1 device, 2 pinned host.  2 * n_frames <= 1024;
 * boxsize a multiple of 8.  A box of width <= 0 (the reference's cv2.resize raises on it) counts as a missing hand.
 * wait: HandMat n x 42 x 3 float64 (rows 0-20 left hand, 21-41 right hand; a coordinate of exactly 0 means "missing"
 * -- a missing hand keeps the scores Batch_hand finds on its grey crop).  hand_s must not be used by other calls
 * while a batch is in flight.                                                                             */
int opb_hand_track_submit(opb_session* hand_s, const uint8_t* frames_bgr, int where, int n_frames, int height, int width,
                          const double* host_poses, int boxsize);
int opb_hand_track_wait(opb_session* hand_s, double* hand_mats);
/* the 2n crops of the last hand-track batch, (2n, boxsize, boxsize, 3) uint8, slot 2f the left hand of frame f (parity
 * tests); valid until the session runs other work.                                                   */
int opb_hand_track_crops(opb_session* hand_s, uint8_t* host_crops);
/* Host only (no device call): the two boxes of one pose (pose54 = 18 x 3) in a height x width frame, computed by the
 * same function as the device -- boxes8 = [left, right] x [x, y, w, valid]; (0, 0, 0, 0) when a joint is missing.  */
int opb_hand_track_boxes(const double* pose54, int height, int width, int* boxes8);
/* ---- Batch_body_extraction + Batch_hand_extraction (srcmx/Batch_motion_Estimation.py:19-112) in one pass -----------
 * For n_frames ROI-cropped frames (n, height, width, 3) uint8, uploaded once: Batch_body on them (as
 * opb_batch_body_submit_u8 with g_scale), the person with the largest left-shoulder x and its 18 body rows (body_pose,
 * :86-105), both hand boxes derived from those rows exactly as from the saved MotionMat (HandImageDataset.__getitem__,
 * srcmx/Batch_model.py:68-104: a joint is missing when x + y + score == 0), the crops cv2.resize(crop, (boxsize,
 * boxsize), INTER_CUBIC) cut from the frames already on the device -- the left one mirrored, a uniform 128 image where a
 * hand is missing --, Batch_hand on all 2n crops and the key points moved back to ROI coordinates (:41-56).  Both tracks
 * equal those of the two jobs run one after the other.  `where`: 0 pageable host, 1 device, 2 pinned host.
 * 1 <= n_frames <= 64; boxsize a positive multiple of 8; body_s on a body network and hand_s on a hand network of the
 * same context.  hand_s must not be used by other calls while a batch is in flight.
 * wait: MotionMat n x 18 x 3 and HandMat n x 42 x 3 float64 (HandMat rows 0-20 left hand, 21-41 right hand; a
 * coordinate of exactly 0 means "missing"; a missing hand -- a missing joint, or a box of width <= 0, on which the
 * reference's cv2.resize raises -- keeps the scores Batch_hand finds on its grey crop).  frame_status (optional): n
 * ints, OPB_OK or OPB_ERR_SUBSET_INDEX per frame; returns the first non-OK status like opb_body_wait_batch.
 * opb_hand_track_crops(hand_s) returns the crops of the last batch.                                                  */
int opb_batch_pose_submit(opb_session* body_s, opb_session* hand_s, const uint8_t* frames_bgr, int where, int n_frames,
                          int height, int width, double g_scale, int boxsize);
int opb_batch_pose_wait(opb_session* body_s, double* motion_mats /* n x 18 x 3 */, double* hand_mats /* n x 42 x 3 */,
                        int* frame_status);
/* ---- every person on the batched estimators -----------------------------------------------------------------------
 * opb_batch_pose_submit's sequence for EVERY person Batch_body finds, not just the one with the largest left-shoulder x:
 * per frame one 60 x 3 float64 record per subset row, in subset order -- rows 0-17 candidate[subset[p][k]][:3], rows
 * 18-38 / 39-59 the left / right HandMat rows Batch_hand_extraction would derive from those body rows (boxes as
 * HandImageDataset.__getitem__, crops cv2.resize(crop, (boxsize, boxsize), INTER_CUBIC), the left one mirrored, grey
 * for a missing hand, Batch_hand, :41-56 back to ROI coordinates).  Every person gets both crops; a missing hand -- a
 * missing joint, or a box of width <= 0 -- keeps the scores Batch_hand finds on its grey crop, with coordinates 0.
 * Arguments and checks as opb_batch_pose_submit.  The crops run in fixed chunks through one Batch_hand plan, so memory
 * does not depend on the number of persons.  Results: opb_pose_every_wait / _wait_tracked / _fetch / _fetch_ids.
 * hand_s must not be used by other calls while a batch is in flight.                                               */
int opb_batch_pose_every_submit(opb_session* body_s, opb_session* hand_s, const uint8_t* frames_bgr, int where,
                                int n_frames, int height, int width, double g_scale, int boxsize);

/* blurred heat maps of the last batched-estimator call: (n, 19 | 22, height, width) planar fp32; the
 * un-blurred maps and the PAFs come from opb_body_maps / opb_hand_maps.                             */
int opb_batch_maps(opb_session* s, float* host_blurred_heat);
/* Debug: the bf16 net input of the last batched-estimator call, (n, hp, wp, 3) bit patterns: the resized frames (a
 * Batch_hand crop is not resized) minus 0.5, zero padding to multiples of 8 (hp, wp as O.batch_size_pad gives them).  */
int opb_batch_debug_input(opb_session* s, uint16_t* host_dst);

/* ---- stage-level entry points on DEVICE buffers (parity tests, per-stage benches) ------------- */
/* src/body.py:38-41 + src/util.py:12-32: cubic resize by `multiplier`, pad right/bottom with 128 to a
 * multiple of 8.  out_u8: (hp, wp, 3) uint8.  Query the sizes first with opb_scale_dims.             */
int opb_scale_dims(int height, int width, double scale, int* h, int* w, int* hp, int* wp);
int opb_preprocess(opb_context* ctx, const uint8_t* dev_img, int height, int width, double scale,
                   uint8_t* dev_out_u8);
/* src/model.py:106-133 / 197-214 on an already preprocessed uint8 padded image batch
 * (n, hp, wp, 3).  Outputs are fp32 NHWC with channel strides 40 (PAF, 38 used), 24 (heat, 19 used)
 * for the body net, 24 (22 used) for the hand net (paf_out is ignored for the hand net).            */
int opb_net_forward(opb_session* s, const uint8_t* dev_in_u8, int n, int hp, int wp, float* dev_paf_out,
                    float* dev_heat_out);
/* src/body.py:54-68: x8 cubic, crop, cubic resize to (H,W), average over scales.
 * maps[i]: fp32 NHWC (ho_i, wo_i, cstride) net output of scale i; out: planar fp32 (C, H, W).        */
int opb_upsample_avg(opb_context* ctx, const float* const* dev_maps, const double* scale_search, int n_scales,
                     int channels, int cstride, int height, int width, float* dev_out);
/* src/body.py:70-94: Gaussian sigma=3 + 4-neighbour NMS + threshold on parts 0..17 of a planar
 * (>=18, H, W) fp32 map.  candidates: (capacity, 4) float64 device buffer (x, y, raw score, id) in the
 * reference's order; part_begin: 19 ints.  Returns OPB_ERR_CAPACITY (with *n set) if it overflowed.  */
int opb_find_peaks(opb_context* ctx, const float* dev_heat, int height, int width, double thre1,
                   double* dev_candidates, int capacity, int* host_part_begin19, int* n);
/* srcmx/utilmx.py:230-241 + srcmx/Batch_model.py:185-194: peaks of an already blurred planar (>=18, H, W) fp32 map,
 * threshold compared in float32, scored with the blurred value.  Same outputs as opb_find_peaks.      */
int opb_find_peaks_blurred(opb_context* ctx, const float* dev_blurred, int height, int width, double thre1,
                           double* dev_candidates, int capacity, int* host_part_begin19, int* n_candidates);
/* src/body.py:96-212 on device maps + the candidates of opb_find_peaks.  Results to host.           */
int opb_group_limbs(opb_context* ctx, const float* dev_paf, int height, int width, const double* dev_candidates,
                    const int* host_part_begin19, double thre2, double* host_subset, int subset_capacity,
                    int* n_subset, double* host_connections /* optional 19*conn_cap*5 */, int conn_capacity,
                    int* host_conn_count19 /* optional */);
/* Measurement helper for BASELINE.json's second metric ("PAF-grouping ms/frame"): times `iters` repetitions of
 * src/body.py:70-212 (Gaussian + NMS + peak ordering + PAF scoring + matching + assembly) on resident device maps
 * with CUDA events, buffers allocated once.                                                            */
int opb_bench_grouping(opb_context* ctx, const float* dev_heat, const float* dev_paf, int height, int width,
                       int iters, float* ms_per_frame, int* n_candidate, int* n_subset);
/* srcmx/MotionEstimation.py:141-162 + src/util.py:133-201 on host-provided body results of one frame: body rows of
 * PoseMat (host_pose180 = 60 x 3, hand rows zero) and the two hand boxes (host_boxes8 = [left, right] x
 * [x, y, w, valid]) -- the device kernel of the opb_pose_* pipeline, for parity tests.                 */
int opb_pose_select(opb_context* ctx, const double* host_candidates, int n_candidates, const double* host_subset,
                    int n_subset, int height, int width, double* host_pose180, int* host_boxes8);
/* The rows-and-boxes kernel of the opb_pose_every_* pipeline on host-provided body results of one frame (parity tests):
 * host_records = n_subset x 60 x 3 (body rows, hand rows zero); host_boxes = 2 * n_subset x [x, y, w, is_left,
 * record], the boxes util.handDetect returns in its order, rows past the box count all -1.                        */
int opb_pose_every_select(opb_context* ctx, const double* host_candidates, int n_candidates, const double* host_subset,
                          int n_subset, int height, int width, double* host_records, int* host_boxes);
/* The same for opb_batch_pose_every_*: host_boxes = 2 * n_subset x [x, y, w, valid, is_left, record], both slots of
 * every person (left first) in person order; (0, 0, 0, 0) for a hand with a missing joint, valid 0 for a box of width
 * <= 0.                                                                                                              */
int opb_batch_pose_every_select(opb_context* ctx, const double* host_candidates, int n_candidates,
                                const double* host_subset, int n_subset, int height, int width, double* host_records,
                                int* host_boxes);
/* src/hand.py:59-75 on a planar (>=21, h, w) fp32 device map -> 21x3 float64 host array.            */
int opb_hand_peaks(opb_context* ctx, const float* dev_heat, int height, int width, double thre, double* host_peaks);
/* Debug: the hand post-processing launches of one geometry on planar fp32 device maps, crop c's 21 key-point planes
 * at dev_maps + c * chan_stride planes.  mode 0 (Hand, threshold 0.03 on the sigma=3 smoothing): sides == NULL runs
 * the equal-size launch on n_crops maps of height x width; otherwise the list launch, crop c of side sides[c] (0 = no
 * crop, zero key points), planes at pitch max(sides)^2 (height and width are ignored).  mode 1 (Batch_hand, threshold
 * 0.035f on the maps as given).  Optional device outputs: dev_smoothed (mode 0 equal size) the float64 smoothed
 * planes, dev_labels the component labels (root = smallest raster index of the component, -1 off the mask),
 * dev_sums the sums plane, each n_crops * 21 planes at the geometry's pitch.  flags & 1: every component counts as a
 * contender of the component choice, and dev_sums holds numpy's sum of each component at its root.
 * host_peaks: n_crops * 21 * 3 doubles (x, y, score). */
int opb_hand_debug_post(opb_context* ctx, const float* dev_maps, int n_crops, int chan_stride, const int* sides, int height,
                        int width, int mode, int flags, double* dev_smoothed, int* dev_labels, double* dev_sums,
                        double* host_peaks);
/* Host only (no device call): np.sum of n contiguous float32 (is_f32) or float64 values, computed by the pairwise
 * summation the device's component choice uses; *out = the result (float32 results widened). */
int opb_debug_pairwise_sum(const void* values, long long n, int is_f32, double* out);

/* Debug: the float64 Gaussian-smoothed maps (parts, H, W) the NMS compares, for bit-exactness tests. */
int opb_smooth_debug(opb_context* ctx, const float* dev_heat, int parts, int height, int width, double* dev_smoothed);

/* Debug/cross-check: generic convolution on NHWC bf16 device tensors through either the tcgen05
 * implicit-GEMM path the networks use (impl = 0), the scalar reference kernel (impl = 1), or a specific
 * tensor-core variant (2 = per-tap tiles, 3 / 4 = patch-resident MODE 0 / 1, 5 = CTA pair, 6 = CTA pair in the
 * wide-pixel pooled form the networks use for conv1_2: cin = cout = 64, k = 3, pool != 0).  weight is host OIHW fp32.
 * out_fp32 != 0 writes fp32.  pool != 0 fuses a 2x2/2 max-pool (impl 0 only).                         */
int opb_conv2d(opb_context* ctx, const void* dev_in_bf16, int n, int h, int w, int cin, const float* weight,
               const float* bias, int cout, int k, int relu, int pool, int out_fp32, void* dev_out, int impl);

/* Debug: one CNN execution plan, step by step (layer-by-layer tests).
 * plan      : builds (or finds) the session's plan for n_scales input shapes, shapes[4 * i ..] = {n, hp, wp, in_elem}
 *             (in_elem 1: uint8 pixels, 2: bf16 values as the batched estimators feed them); *n_steps = its steps.  Later
 *             calls refer to this plan (it is looked up again by its shapes, so it may be rebuilt, never dangles).
 * set_input : copies scale `scale`'s input, (n, hp, wp, 3) elements of in_elem bytes, from device memory.
 * info      : what step i computes (no device work).
 * step      : runs step i alone on the session's stream, waits for it, and fills *info.
 * read      : copies a view of step i (problem p; which 0 = input, 1 = output) densely into dev_dst as (n, h, w, c)
 *             elements of `elem` bytes, and waits for the copy.
 * run       : runs every step back to back as opb_net_forward does, then waits once.                               */
#define OPB_DEBUG_MAX_PROBLEMS 8
#define OPB_STEP_CONV_FIRST 0  /* conv1_1 on the CUDA-core / mma.sync path                                    */
#define OPB_STEP_CONV 1        /* a grouped tensor-core convolution launch                                    */
#define OPB_STEP_TAIL 2        /* fused 1x1 -> ReLU -> 1x1 tail, 128-channel intermediate (Mconv6 -> Mconv7)  */
#define OPB_STEP_TAIL_WIDE 3   /* fused tail with a 512-channel intermediate (conv5_4 -> conv5_5, conv6_1 -> conv6_2) */
#define OPB_STEP_POOL 4        /* stand-alone 2x2 max-pool (OPB_NO_FUSE_POOL=1)                               */
typedef struct opb_debug_view {
    int n, h, w, c, cstride, coff, elem;
} opb_debug_view;
typedef struct opb_debug_step {
    int kind;                  /* OPB_STEP_*                                                                   */
    int n_problems;
    int block_n;               /* N tile that runs (tensor-core launches)                                       */
    int pool;                  /* fused 2x2 max-pool                                                            */
    int wide;                  /* conv1_2 ran in the wide-pixel form (the views are those of the plain layer)   */
    int pair;                  /* CTA-pair kernel                                                               */
    int half_tiles;            /* CTA pair: 16 x 8 tiles                                                        */
    int weights_resident;      /* CTA pair: one weight set kept in shared memory for the whole kernel          */
    char name[64];             /* the step's profile name (conv_tc128:..., conv_tc64:..., conv_tail:..., ...) */
    char layer[OPB_DEBUG_MAX_PROBLEMS][32];
    char layer2[OPB_DEBUG_MAX_PROBLEMS][32];   /* second layer of a fused tail, else ""                       */
    int scale[OPB_DEBUG_MAX_PROBLEMS];
    opb_debug_view in[OPB_DEBUG_MAX_PROBLEMS], out[OPB_DEBUG_MAX_PROBLEMS];
} opb_debug_step;
int opb_net_debug_plan(opb_session* s, int n_scales, const int* shapes, int* n_steps);
int opb_net_debug_set_input(opb_session* s, int scale, const void* dev_src);
int opb_net_debug_info(opb_session* s, int i, opb_debug_step* info);
int opb_net_debug_step(opb_session* s, int i, opb_debug_step* info);
int opb_net_debug_read(opb_session* s, int i, int problem, int which, void* dev_dst);
int opb_net_debug_run(opb_session* s);

/* Post-processing of Body (mode 0: scale_search, 1..8 scales) and Batch_body (mode 1: g_scale, one scale) on net
 * outputs the caller supplies, through the frame plan a real call of that geometry uses: the same tile bounds, fused
 * peak kernel, composite PAF sampling and grouping, only the upload, the front end and the CNN are skipped.
 * post_dims (host only): ho_wo[2 * i], ho_wo[2 * i + 1] = the net output size of scale i; *fused = 1 when the peak
 *   kernel evaluates the heat maps from the net outputs, 0 when the plan materialises them first.
 * post_submit: heat[i] (n, ho, wo, 24) and paf[i] (n, ho, wo, 40) fp32 host arrays per scale (19 / 38 channels used).
 *   Results through opb_body_wait_batch / opb_body_fetch_frame; the maps through opb_body_maps / opb_batch_maps.
 * part_begin (after a wait, any body batch): first candidate row of each of the 18 parts of a frame, and the total. */
int opb_body_debug_post_dims(int height, int width, const double* scales, int n_scales, int mode, int* ho_wo, int* fused);
int opb_body_debug_post_submit(opb_session* s, int n_frames, int height, int width, const double* scales, int n_scales,
                               int mode, const float* const* heat, const float* const* paf);
int opb_body_debug_part_begin(opb_session* s, int frame, int* part_begin19);

/* Host only (no device call): the wide-pixel weights of a 64 -> 64 channel 3x3 layer (src/model.py:36 conv1_2) as the
 * library packs them at opb_net_finalize.  weight: [64][64][3][3] fp32, bias [64]  ->  w_wide [128][9][128] bf16 bit
 * patterns (output column = parity_out * 64 + cout; K index = (dy * 3 + di) * 128 + parity_in * 64 + cin, di the tap in
 * units of column PAIRS), b_wide [128].  Lets a CPU test prove the re-described layer equals the original one.        */
int opb_wide_pool_weights(const float* weight, const float* bias, unsigned short* w_wide, float* b_wide);

/* Host only (no device call): the resampling tables the library builds on the host and its kernels apply.
 * opb_debug_resize_taps: cv2's INTER_CUBIC taps for one axis (first tap index, may lie outside the source: taps are
 *   clamped when used; 4 float32 coefficients per destination index) -- src/body.py:38,55,57.
 * opb_debug_composite_taps: the per-axis operator of "x8 cubic upsample, crop to n_resized, cubic resize to n_orig"
 *   (src/body.py:55-57) as first source index + 6 float32 weights per destination index.
 * opb_debug_resize_dsize: cv2's destination size for a scale factor (round half to even).
 * opb_debug_hand_track_taps: the taps opb_hand_track_submit's tables hold for a side x side crop resized to boxsize
 *   (boxsize entries of first / coef4).                                                                             */
int opb_debug_resize_taps(int src, int dst, double scale, int* first, float* coef4);
int opb_debug_hand_track_taps(int side, int boxsize, int* first, float* coef4);
int opb_debug_composite_taps(int n_net, int n_resized, int n_orig, int* first, float* w6);
int opb_debug_resize_dsize(int n, double f);
/* The same for Batch_body / Batch_hand, whose resizes are torch's F.interpolate(mode="bicubic") on float32:
 * opb_debug_batch_resize_taps: the front end's taps, F.interpolate(scale_factor=scale_factor), or size mode (dst
 *   given) when scale_factor <= 0.
 * opb_debug_batch_composite_taps: the map side, F.interpolate(scale_factor=8), crop to n_resized,
 *   F.interpolate(size=n_orig).                                                                                     */
int opb_debug_batch_resize_taps(int src, int dst, double scale_factor, int* first, float* coef4);
int opb_debug_batch_composite_taps(int n_net, int n_resized, int n_orig, int* first, float* w6);

/* Host only (no device call): the tile list of the CTA-pair convolution kernel for one problem of n images of h x w
 * pixels, exactly as the kernel decodes it -- 8 ints per (pair, cluster rank): image, x0, y0, n0, real (0 = padding tile,
 * computed but never stored), halves (bit h: 128-pixel half h holds pixels), vsplit (0 = halves side by side 8 x 16,
 * 1 = stacked 16 x 8), full_cost.  small != 0: the 16 x 8 tiles of launches that fill few SMs.  For the CPU test of
 * the tiling (every pixel stored exactly once, both tiles of a pair share one orientation).  *written = entries.     */
int opb_debug_pair_tiles(int n, int h, int w, int n_tiles_n, int small, int* out, int cap, int* written);

/* ---- MJPG frames decoded on the device ------------------------------------------------------------------------
 * A decoded frame equals cv2.imdecode(packet, cv2.IMREAD_COLOR) bit for bit (libjpeg-turbo's ISLOW IDCT, fancy
 * upsampling and YCbCr -> BGR tables), cropped like numpy's frame[y0:y1, x0:x1].  Baseline / extended sequential
 * Huffman JPEG, 8-bit, one scan: grey, or YCbCr 4:4:4, 4:2:2, 4:2:0.  Other packets are not decoded here
 * (OPB_JPEG_FALLBACK): the caller decodes them and puts the frame in place with opb_jpeg_upload.
 *
 * opb_jpeg_submit: n packets, packet i = packed[offsets[i] .. offsets[i + 1]) in host memory (where 0 pageable or 2
 *   pinned: both are read the same way -- the host parses and destuffs every packet into the session's own pinned
 *   buffer and uploads from there, so pinned packets gain nothing), are parsed on the host and decoded on the session's
 *   stream, so the session's next submit with where = 1
 *   reads them in stream order.  roi = {x0, y0, x1, y1} (Python slice ends) or NULL for the whole frame; every packet
 *   of a batch must have the same frame size.  flags[n] gets what the host already knows: OPB_JPEG_FALLBACK, or
 *   OPB_JPEG_CORRUPT for restart markers that do not match the header.  *dev_frames: (n, height, width, 3) uint8 BGR
 *   device frames, valid until the session's next opb_jpeg_submit.  The call does not wait for the stream; it waits
 *   only for the upload of the session's previous batch before reusing its pinned buffers.
 * opb_jpeg_upload: copies the host frame (height, width, 3) of a packet decoded elsewhere into slot `index`.
 * opb_jpeg_fetch: waits for the stream and copies the n frames to host memory.
 * opb_jpeg_status: waits for the decode and gives flags[n]: the submit's flags | OPB_JPEG_CORRUPT for entropy data
 *   the device could not decode consistently (a bad Huffman code, a segment that runs out or has data left over).
 * opb_jpeg_decode_host (host only): the same decoder on the CPU, for one packet.  *height / *width / *status are set
 *   first (0 x 0 when no frame header was read); the frame is written when out != NULL and *status == 0 after
 *   parsing (OPB_ERR_CAPACITY when out_bytes is short).  Malformed headers return OPB_ERR_INVALID.             */
#define OPB_JPEG_FALLBACK 1
#define OPB_JPEG_CORRUPT 2
int opb_jpeg_submit(opb_session* s, const uint8_t* packed, const int64_t* offsets, int where, int n, const int* roi,
                    int* flags, uint8_t** dev_frames, int* height, int* width);
int opb_jpeg_upload(opb_session* s, int index, const uint8_t* host_frame);
int opb_jpeg_fetch(opb_session* s, uint8_t* host_out);
int opb_jpeg_status(opb_session* s, int* flags);
int opb_jpeg_decode_host(const uint8_t* packet, int64_t size, const int* roi, uint8_t* out, int64_t out_bytes,
                         int* height, int* width, int* status);

#ifdef __cplusplus
}
#endif
#endif /* OPENPOSE_B200_H_ */
