// Baseline JPEG decoding on the device (jpeg.cu): the interface api.cu's opb_jpeg_* entries call.
#pragma once
#include "opb_common.cuh"

namespace opb {

// per-frame flags of a decoded batch (opb_jpeg_submit / opb_jpeg_status)
constexpr int kJpegFallback = 1;   // not decoded on the device: unsupported or unreadable header (known at submit)
constexpr int kJpegCorrupt = 2;    // entropy data inconsistent with the header (a bad code, a segment that runs out)

struct JpegBatch;                  // one session's decode buffers (pinned parameters, device planes and frames)
void jpeg_batch_free(JpegBatch* jb);

// Parses the n packets (packed, offsets[n + 1]) on the host and enqueues their decode on `st`.  flags[n] gets
// kJpegFallback / kJpegCorrupt for packets the host already knows the device will not decode.  *dev receives the
// (n, h, w, 3) BGR frames, ROI-cropped like numpy's frame[y0:y1, x0:x1] (roi = {x0, y0, x1, y1}, or null).
// Returns the kernels launched.
int jpeg_submit(JpegBatch*& jb, int device, cudaStream_t st, const uint8_t* packed, const int64_t* offsets, int n,
                const int* roi, int* flags, uint8_t** dev, int* h, int* w);
// copies one host frame (h, w, 3) into slot `index` of the last batch (a packet decoded elsewhere)
void jpeg_upload(JpegBatch* jb, cudaStream_t st, int index, const uint8_t* frame);
// waits for the last batch; its frames to host memory
void jpeg_fetch(JpegBatch* jb, cudaStream_t st, uint8_t* host);
// waits for the last batch's device flags; flags[n] = host flags | device flags
void jpeg_status(JpegBatch* jb, int* flags);
// the whole decoder on the CPU: same parser, same per-block and per-pixel arithmetic
void jpeg_decode_host(const uint8_t* packet, int64_t size, const int* roi, uint8_t* out, int64_t out_bytes, int* h,
                      int* w, int* status);

}  // namespace opb
