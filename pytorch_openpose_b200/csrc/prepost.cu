// Streaming kernels either side of the CNN.
//
//   preprocess   : src/body.py:38-39 + src/util.py:12-32 -- cv2.resize(INTER_CUBIC) of the uint8 BGR frame by
//                  `multiplier`, then pad right/bottom with 128 to a multiple of 8.  The arithmetic follows
//                  OpenCV's open-source resize exactly (11-bit fixed-point taps, int32 horizontal pass, float
//                  vertical pass accumulated S3,S2,S1,S0 with separate multiply and add, integer pass for the
//                  last (3*w) % 8 elements of every row), so it is bit-identical to cv2 with IPP disabled
//                  (see oracle/openpose_oracle.py::resize_cubic_u8).  The /256-0.5 normalisation and the
//                  HWC->NCHW transpose of src/body.py:40 are folded into the first convolution.
//   upsample_avg : src/body.py:54-68 / src/hand.py:52-57 -- x8 cubic upsample, crop of the padding, cubic
//                  resize to the frame size and the cross-scale average.  Both cubic passes are linear and
//                  separable, so each axis collapses into one banded operator with <= 6 taps per output
//                  index (tables built on the host in float64, oracle: composite_upsample_matrix).
//                  Pass 1 applies the x operator per scale into an L2-resident (C, ho, W) scratch, pass 2
//                  applies the y operators of all scales, averages and writes the planar (C, H, W) map once.
#include "opb_common.cuh"

namespace opb {
namespace {

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// one thread per output PIXEL (y, x) of the padded image: the three channels share the tap indices and weights
__global__ void __launch_bounds__(128) preprocess_kernel(const uint8_t* __restrict__ img, int H, int W,
                                                         uint8_t* __restrict__ out, int h, int w, int hp, int wp,
                                                         const int* __restrict__ xf, const short* __restrict__ xc,
                                                         const int* __restrict__ yf, const short* __restrict__ yc,
                                                         size_t img_stride, size_t out_stride) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y;
    if (x >= wp) return;
    img += blockIdx.z * img_stride;
    out += blockIdx.z * out_stride;
    uint8_t* o = out + ((size_t)y * wp + x) * 3;
    if (y >= h || x >= w) {
        o[0] = o[1] = o[2] = 128;                               // padValue, src/body.py:29
        return;
    }
    const int x0 = xf[x], y0 = yf[y];
    int cx[4], wx[4];
    const short4 xw4 = *(const short4*)(xc + x * 4);
    wx[0] = xw4.x; wx[1] = xw4.y; wx[2] = xw4.z; wx[3] = xw4.w;
#pragma unroll
    for (int j = 0; j < 4; ++j) cx[j] = clampi(x0 + j, 0, W - 1) * 3;
    int hor[4][3];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint8_t* row = img + (size_t)clampi(y0 + k, 0, H - 1) * W * 3;
        int s0 = 0, s1 = 0, s2 = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint8_t* px = row + cx[j];
            s0 += (int)__ldg(px) * wx[j];
            s1 += (int)__ldg(px + 1) * wx[j];
            s2 += (int)__ldg(px + 2) * wx[j];
        }
        hor[k][0] = s0; hor[k][1] = s1; hor[k][2] = s2;
    }
    const short4 yw4 = *(const short4*)(yc + y * 4);
    const int wyi[4] = {yw4.x, yw4.y, yw4.z, yw4.w};
    const float sc = 1.0f / (2048.0f * 2048.0f);
    float wyf[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) wyf[k] = __fmul_rn((float)wyi[k], sc);
    const int nvec = ((w * 3) / 8) * 8;                         // OpenCV: 8-lane SIMD body, scalar tail
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        int r;
        if (x * 3 + c < nvec) {
            float acc = __fmul_rn((float)hor[3][c], wyf[3]);
#pragma unroll
            for (int k = 2; k >= 0; --k) acc = __fadd_rn(acc, __fmul_rn((float)hor[k][c], wyf[k]));
            r = __float2int_rn(acc);
        } else {
            long long s = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k) s += (long long)hor[k][c] * (long long)wyi[k];
            r = (int)((s + (1ll << 21)) >> 22);
        }
        o[c] = (uint8_t)clampi(r, 0, 255);
    }
}

// pass 1: tmp[c][r][x] = sum_k xw[x][k] * src[r][xfirst[x]+k][c]      (one scale)
// one thread = one output column x and FOUR consecutive channels (one float4 per tap from the NHWC source)
__global__ void upsample_x_kernel(const float* __restrict__ src, int ho, int wo, int cstride, int C, int W,
                                  const int* __restrict__ xfirst, const float* __restrict__ xw,
                                  float* __restrict__ tmp) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int r = blockIdx.y;
    const int cq_per_img = (C + 3) >> 2;
    const int img = blockIdx.z / cq_per_img, cq = blockIdx.z - img * cq_per_img;
    if (x >= W) return;
    const int f = xfirst[x];
    const float* s = src + (((size_t)img * ho + r) * wo) * cstride + cq * 4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int k = 0; k < kUpTaps; ++k) {
        const int col = min(f + k, wo - 1);                     // weights beyond the footprint are zero
        const float wk = xw[x * kUpTaps + k];
        const float4 v = *(const float4*)(s + (size_t)col * cstride);
        acc.x = fmaf(wk, v.x, acc.x);
        acc.y = fmaf(wk, v.y, acc.y);
        acc.z = fmaf(wk, v.z, acc.z);
        acc.w = fmaf(wk, v.w, acc.w);
    }
    const float av[4] = {acc.x, acc.y, acc.z, acc.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int ch = cq * 4 + j;
        if (ch < C) tmp[(((size_t)img * C + ch) * ho + r) * W + x] = av[j];
    }
}

struct UpYParams {
    const float* tmp[kMaxScales];     // (C, ho, W) per scale
    const int* yfirst[kMaxScales];
    const float* yw[kMaxScales];      // 1/n_scales folded in
    int ho[kMaxScales];
    int n_scales;
};

// pass 2 (generic shapes): out[c][y][x] = chain over scales s, taps k of fmaf(yw_s[y][k], tmp_s[c][yfirst_s[y]+k][x], .)
// -- the same chain as the register-blocked kernel below and as composite.cuh (zero-weight strip rows are no-ops)
template <int VEC>
__global__ void upsample_y_kernel(const __grid_constant__ UpYParams p, int C, int H, int W, float* __restrict__ out) {
    const int xv = blockIdx.x * blockDim.x + threadIdx.x;
    const int x = xv * VEC;
    const int y = blockIdx.y;
    const int c = blockIdx.z;
    if (x >= W) return;
    float acc[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) acc[v] = 0.f;
    for (int s = 0; s < p.n_scales; ++s) {
        const int f = p.yfirst[s][y];
        const int ho = p.ho[s];
        const float* t = p.tmp[s] + (size_t)c * ho * W + x;
#pragma unroll
        for (int k = 0; k < kUpTaps; ++k) {
            const float wgt = p.yw[s][y * kUpTaps + k];
            const int r = min(f + k, ho - 1);
            if (VEC == 4) {
                const float4 q = *(const float4*)(t + (size_t)r * W);
                acc[0] = fmaf(wgt, q.x, acc[0]);
                acc[1 % VEC] = fmaf(wgt, q.y, acc[1 % VEC]);
                acc[2 % VEC] = fmaf(wgt, q.z, acc[2 % VEC]);
                acc[3 % VEC] = fmaf(wgt, q.w, acc[3 % VEC]);
            } else {
                acc[0] = fmaf(wgt, t[(size_t)r * W], acc[0]);
            }
        }
    }
    float* o = out + ((size_t)c * H + y) * W + x;
    if (VEC == 4)
        *(float4*)o = make_float4(acc[0], acc[1 % VEC], acc[2 % VEC], acc[3 % VEC]);
    else
        o[0] = acc[0];
}

// pass 2, register-blocked: one thread produces a 16-row x 4-column strip of one channel plane.  It walks the source
// rows its strip touches once (a float4 each) and scatters them into 16 accumulators with the dense per-strip weight
// table built on the host (1/n_scales folded in), so every scratch element is read ~2x instead of 24x.
constexpr int kTY = kUpStrip;
struct UpYBlocked {
    const float* tmp[kMaxScales];
    const int* first[kMaxScales];      // [n_yblocks]            first source row of the strip
    const int* rows[kMaxScales];       // [n_yblocks]            source rows the strip touches
    const float* w[kMaxScales];        // [n_yblocks][rs][16]    weight of source row r for output row yy
    int ho[kMaxScales], rs[kMaxScales];
    int n_scales;
};
constexpr int kMaxStripRows = 24;           // source rows one 16-row strip may touch per scale (host falls back otherwise)
__global__ void __launch_bounds__(128) upsample_y_blocked_kernel(const __grid_constant__ UpYBlocked p, int CT, int H,
                                                                 int W, float* __restrict__ out) {
    // the strip's weight tables (all scales) go to shared memory once per block: every thread of the block uses the
    // same ones, and as global loads they kept missing L1 behind the streaming row loads (ncu: 15 % L1 hit rate,
    // long-scoreboard stalls 5 per issue)
    __shared__ __align__(16) float sw[kMaxScales][kMaxStripRows * kTY];
    const int yb = blockIdx.y;
    {
        const int tid = threadIdx.y * blockDim.x + threadIdx.x, nthr = blockDim.x * blockDim.y;
        for (int s = 0; s < p.n_scales; ++s) {
            const int n = p.rows[s][yb] * kTY;
            const float* src = p.w[s] + (size_t)yb * p.rs[s] * kTY;
            for (int i = tid; i < n; i += nthr) sw[s][i] = __ldg(src + i);
        }
    }
    __syncthreads();
    const int x = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    const int c = blockIdx.z * blockDim.y + threadIdx.y;
    if (x >= W || c >= CT) return;
    // accumulators as float2 pairs: sm_100's packed FFMA2 (__ffma2_rn) retires two IEEE fp32 FMAs per issue slot --
    // bit-identical to two fmaf, and this kernel is FMA-issue bound (28 FMAs per output element)
    float2 acc[kTY][2];
#pragma unroll
    for (int i = 0; i < kTY; ++i) acc[i][0] = acc[i][1] = make_float2(0.f, 0.f);
    for (int s = 0; s < p.n_scales; ++s) {
        const int f0 = p.first[s][yb], R = p.rows[s][yb];
        const float* t = p.tmp[s] + ((size_t)c * p.ho[s] + f0) * W + x;
        const float4* wt = (const float4*)sw[s];
        // rows are prefetched two ahead: the loads come from L2 / HBM and nothing else in the thread can hide them
        const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
        float4 v0 = R > 0 ? *(const float4*)t : zero4;
        float4 v1 = R > 1 ? *(const float4*)(t + (size_t)W) : zero4;
        for (int r = 0; r < R; ++r) {
            const float4 v = v0;
            v0 = v1;
            v1 = r + 2 < R ? *(const float4*)(t + (size_t)(r + 2) * W) : zero4;
            const float2 vlo = make_float2(v.x, v.y), vhi = make_float2(v.z, v.w);
#pragma unroll
            for (int q = 0; q < kTY / 4; ++q) {
                const float4 w4 = wt[r * (kTY / 4) + q];
                const float ws[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float2 w2 = make_float2(ws[j], ws[j]);
                    acc[q * 4 + j][0] = __ffma2_rn(w2, vlo, acc[q * 4 + j][0]);
                    acc[q * 4 + j][1] = __ffma2_rn(w2, vhi, acc[q * 4 + j][1]);
                }
            }
        }
    }
    float* o = out + ((size_t)c * H + (size_t)yb * kTY) * W + x;
#pragma unroll
    for (int i = 0; i < kTY; ++i)
        if (yb * kTY + i < H)
            *(float4*)(o + (size_t)i * W) = make_float4(acc[i][0].x, acc[i][0].y, acc[i][1].x, acc[i][1].y);
}

// ---- ragged hand crops (the per-frame caller, srcmx/MotionEstimation.py:163-194): every slot of the batch is a square
// crop of its own size taken from a frame that is already on the device.  The tap tables of every possible size sit in
// one slab (built on the host with the same functions as the single-size path); `index` holds, per (size, scale), the
// byte offsets of {preprocess first, preprocess coef, upsample first, upsample x weights, upsample y weights (1/n_scales
// folded in)}.
__device__ __forceinline__ const uint8_t* ragged_table(const RaggedTables& t, int w, int scale, int which) {
    return t.slab + t.index[((size_t)w * t.n_scales + scale) * 5 + which];
}

// Hand.__call__'s cv2.resize of the crop (src/hand.py:38) for every slot, reading the crop -- mirrored for left hands,
// cv2.flip(crop, 1) at srcmx/MotionEstimation.py:191 -- straight from the frame.  Arithmetic as preprocess_kernel.
// kPacked: slot i's crop is its own dense w x w image at byte offset offsets[i] of `frames` (Hand()(list of crops));
// the box then only carries the side (x = y = 0, not mirrored).
template <bool kPacked>
__global__ void __launch_bounds__(128) preprocess_ragged_kernel(const uint8_t* __restrict__ frames, int H, int W,
                                                                const size_t* __restrict__ offsets,
                                                                const HandBox* __restrict__ boxes, uint8_t* __restrict__ out,
                                                                int S, int scale, const RaggedTables tabs) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y;
    if (x >= S) return;
    const HandBox b = boxes[blockIdx.z];
    uint8_t* o = out + (((size_t)blockIdx.z * S + y) * S + x) * 3;
    if (!b.valid) {
        o[0] = o[1] = o[2] = 128;
        return;
    }
    const int w = b.w;
    const int* xf = (const int*)ragged_table(tabs, w, scale, 0);
    const short* xc = (const short*)ragged_table(tabs, w, scale, 1);
    const uint8_t* img = kPacked ? frames + offsets[blockIdx.z] : frames + (size_t)b.frame * H * W * 3;
    const int pitch = kPacked ? w : W;
    const int x0 = xf[x], y0 = xf[y];                            // square crops: one table for both axes
    int cx[4], wx[4];
    const short4 xw4 = *(const short4*)(xc + x * 4);
    wx[0] = xw4.x; wx[1] = xw4.y; wx[2] = xw4.z; wx[3] = xw4.w;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int c = clampi(x0 + j, 0, w - 1);
        cx[j] = (b.x + (b.left ? w - 1 - c : c)) * 3;
    }
    int hor[4][3];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint8_t* row = img + (size_t)(b.y + clampi(y0 + k, 0, w - 1)) * pitch * 3;
        int s0 = 0, s1 = 0, s2 = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint8_t* px = row + cx[j];
            s0 += (int)__ldg(px) * wx[j];
            s1 += (int)__ldg(px + 1) * wx[j];
            s2 += (int)__ldg(px + 2) * wx[j];
        }
        hor[k][0] = s0; hor[k][1] = s1; hor[k][2] = s2;
    }
    const short4 yw4 = *(const short4*)(xc + y * 4);
    const int wyi[4] = {yw4.x, yw4.y, yw4.z, yw4.w};
    const float sc = 1.0f / (2048.0f * 2048.0f);
    float wyf[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) wyf[k] = __fmul_rn((float)wyi[k], sc);
    const int nvec = ((S * 3) / 8) * 8;                         // OpenCV: 8-lane SIMD body, scalar tail
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        int r;
        if (x * 3 + c < nvec) {
            float acc = __fmul_rn((float)hor[3][c], wyf[3]);
#pragma unroll
            for (int k = 2; k >= 0; --k) acc = __fadd_rn(acc, __fmul_rn((float)hor[k][c], wyf[k]));
            r = __float2int_rn(acc);
        } else {
            long long s = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k) s += (long long)hor[k][c] * (long long)wyi[k];
            r = (int)((s + (1ll << 21)) >> 22);
        }
        o[c] = (uint8_t)clampi(r, 0, 255);
    }
}

// x pass of the ragged upsample: tmp[slot][c][r][x] for x < w_slot (row pitch = w_slot), slot stride = C * ho * wmax
__global__ void upsample_x_ragged_kernel(const float* __restrict__ src, int ho, int wo, int cstride, int C,
                                         const HandBox* __restrict__ boxes, int scale, const RaggedTables tabs, int wmax,
                                         float* __restrict__ tmp) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int r = blockIdx.y;
    const int cq_per = (C + 3) >> 2;
    const int slot = blockIdx.z / cq_per, cq = blockIdx.z - slot * cq_per;
    const HandBox b = boxes[slot];
    if (!b.valid || x >= b.w) return;
    const int w = b.w;
    const int* xfirst = (const int*)ragged_table(tabs, w, scale, 2);
    const float* xw = (const float*)ragged_table(tabs, w, scale, 3);
    const int f = xfirst[x];
    const float* s = src + (((size_t)slot * ho + r) * wo) * cstride + cq * 4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int k = 0; k < kUpTaps; ++k) {
        const int col = min(f + k, wo - 1);
        const float wk = xw[x * kUpTaps + k];
        const float4 v = *(const float4*)(s + (size_t)col * cstride);
        acc.x = fmaf(wk, v.x, acc.x);
        acc.y = fmaf(wk, v.y, acc.y);
        acc.z = fmaf(wk, v.z, acc.z);
        acc.w = fmaf(wk, v.w, acc.w);
    }
    const float av[4] = {acc.x, acc.y, acc.z, acc.w};
    float* t = tmp + (size_t)slot * C * ho * wmax;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int ch = cq * 4 + j;
        if (ch < C) t[((size_t)ch * ho + r) * w + x] = av[j];
    }
}

struct UpYRagged {
    const float* tmp[kMaxScales];     // per scale: [slot][C][ho][w_slot]
    int ho[kMaxScales];
    int n_scales;
};
// y pass: the chain of upsample_y_kernel with per-slot tables; out[slot][c][y][x], plane pitch w_slot, plane stride ps
constexpr int kRaggedRows = 16;       // output rows per block (the grid is sized for the largest possible crop)
__global__ void upsample_y_ragged_kernel(const __grid_constant__ UpYRagged p, int C, const HandBox* __restrict__ boxes,
                                         const RaggedTables tabs, int wmax, size_t ps, float* __restrict__ out) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int slot = blockIdx.z / C, c = blockIdx.z - slot * C;
    const HandBox b = boxes[slot];
    if (!b.valid || x >= b.w) return;
    const int w = b.w;
    for (int y = blockIdx.y * kRaggedRows; y < min(w, ((int)blockIdx.y + 1) * kRaggedRows); ++y) {
        float acc = 0.f;
        for (int s = 0; s < p.n_scales; ++s) {
            const int* yfirst = (const int*)ragged_table(tabs, w, s, 2);
            const float* yw = (const float*)ragged_table(tabs, w, s, 4);
            const int f = yfirst[y];
            const int ho = p.ho[s];
            const float* t = p.tmp[s] + (size_t)slot * C * ho * wmax + (size_t)c * ho * w + x;
#pragma unroll
            for (int k = 0; k < kUpTaps; ++k) {
                const int r = min(f + k, ho - 1);
                acc = fmaf(yw[y * kUpTaps + k], t[(size_t)r * w], acc);
            }
        }
        out[((size_t)slot * C + c) * ps + (size_t)y * w + x] = acc;
    }
}

}  // namespace

void preprocess_launch_batched(const uint8_t* img, int n, int H, int W, uint8_t* out, int h, int w, int hp, int wp,
                               const int* x_first, const short* x_coef, const int* y_first, const short* y_coef,
                               cudaStream_t stream) {
    dim3 grid(cdiv(wp, 128), hp, n);
    preprocess_kernel<<<grid, 128, 0, stream>>>(img, H, W, out, h, w, hp, wp, x_first, x_coef, y_first, y_coef,
                                                (size_t)H * W * 3, (size_t)hp * wp * 3);
    OPB_CUDA(cudaGetLastError());
}

void preprocess_ragged_launch(const uint8_t* frames, int H, int W, const HandBox* boxes, int n_slots, uint8_t* out, int S,
                              int scale, const RaggedTables& tabs, cudaStream_t stream) {
    dim3 grid(cdiv(S, 128), S, n_slots);
    preprocess_ragged_kernel<false><<<grid, 128, 0, stream>>>(frames, H, W, nullptr, boxes, out, S, scale, tabs);
    OPB_CUDA(cudaGetLastError());
}

void preprocess_packed_launch(const uint8_t* packed, const size_t* offsets, const HandBox* boxes, int n_slots, uint8_t* out,
                              int S, int scale, const RaggedTables& tabs, cudaStream_t stream) {
    dim3 grid(cdiv(S, 128), S, n_slots);
    preprocess_ragged_kernel<true><<<grid, 128, 0, stream>>>(packed, 0, 0, offsets, boxes, out, S, scale, tabs);
    OPB_CUDA(cudaGetLastError());
}

// scratch: sum_s n_slots * C * ho_s * wmax floats; out: [n_slots][C] planes at stride wmax * wmax.  The y weights of
// the tables carry 1/n_scales (the same fold as make_up_tables).
void upsample_ragged_launch(const float* const* src, const int* ho, const int* wo, int n_scales, int cstride, int C,
                            const HandBox* boxes, int n_slots, const RaggedTables& tabs, int wmax, float* scratch,
                            float* out_planar, cudaStream_t stream) {
    UpYRagged p;
    memset(&p, 0, sizeof(p));
    p.n_scales = n_scales;
    size_t off = 0;
    for (int s = 0; s < n_scales; ++s) {
        float* tmp = scratch + off;
        off += (size_t)n_slots * C * ho[s] * wmax;
        dim3 grid(cdiv(wmax, 128), ho[s], n_slots * ((C + 3) / 4));
        upsample_x_ragged_kernel<<<grid, 128, 0, stream>>>(src[s], ho[s], wo[s], cstride, C, boxes, s, tabs, wmax, tmp);
        OPB_CUDA(cudaGetLastError());
        p.tmp[s] = tmp;
        p.ho[s] = ho[s];
    }
    dim3 grid(cdiv(wmax, 128), cdiv(wmax, kRaggedRows), n_slots * C);
    upsample_y_ragged_kernel<<<grid, 128, 0, stream>>>(p, C, boxes, tabs, wmax, (size_t)wmax * wmax, out_planar);
    OPB_CUDA(cudaGetLastError());
}

void preprocess_launch(const uint8_t* img, int H, int W, uint8_t* out, int h, int w, int hp, int wp,
                       const int* x_first, const short* x_coef, const int* y_first, const short* y_coef,
                       cudaStream_t stream) {
    preprocess_launch_batched(img, 1, H, W, out, h, w, hp, wp, x_first, x_coef, y_first, y_coef, stream);
}

// scratch: float buffer with room for sum_s n_img*C*ho_s*W elements
void upsample_avg_launch2(const UpsampleScale* scales, int n_scales, int n_img, int C, int H, int W, float* scratch,
                          float* out_planar, cudaStream_t stream) {
    const int CT = n_img * C;                                   // planar output has n_img*C channel planes
    OPB_REQUIRE(n_scales >= 1 && n_scales <= kMaxScales, "upsample_avg: 1..8 scales");
    UpYParams p;
    memset(&p, 0, sizeof(p));
    p.n_scales = n_scales;
    size_t off = 0;
    for (int s = 0; s < n_scales; ++s) {
        const UpsampleScale& u = scales[s];
        float* tmp = scratch + off;
        off += (size_t)CT * u.ho * W;
        OPB_REQUIRE(u.cstride % 4 == 0 && u.cstride >= ((C + 3) / 4) * 4, "upsample: source channel stride must cover C rounded up to 4");
        dim3 grid(cdiv(W, 128), u.ho, n_img * ((C + 3) / 4));
        upsample_x_kernel<<<grid, 128, 0, stream>>>(u.src, u.ho, u.wo, u.cstride, C, W, u.x_first, u.x_w, tmp);
        OPB_CUDA(cudaGetLastError());
        p.tmp[s] = tmp;
        p.yfirst[s] = u.y_first;
        p.yw[s] = u.y_w;
        p.ho[s] = u.ho;
    }
    bool strips_fit = true;
    for (int s = 0; s < n_scales; ++s) strips_fit = strips_fit && scales[s].yb_rs <= kMaxStripRows;
    if (W % 4 == 0 && scales[0].yb_w != nullptr && strips_fit) {
        UpYBlocked b;
        memset(&b, 0, sizeof(b));
        b.n_scales = n_scales;
        for (int s = 0; s < n_scales; ++s) {
            b.tmp[s] = p.tmp[s];
            b.first[s] = scales[s].yb_first;
            b.rows[s] = scales[s].yb_rows;
            b.w[s] = scales[s].yb_w;
            b.ho[s] = scales[s].ho;
            b.rs[s] = scales[s].yb_rs;
        }
        dim3 block(64, 2);
        dim3 grid(cdiv(W / 4, 64), cdiv(H, kTY), cdiv(CT, 2));
        upsample_y_blocked_kernel<<<grid, block, 0, stream>>>(b, CT, H, W, out_planar);
    } else if (W % 4 == 0) {
        dim3 grid(cdiv(W / 4, 64), H, CT);
        upsample_y_kernel<4><<<grid, 64, 0, stream>>>(p, CT, H, W, out_planar);
    } else {
        dim3 grid(cdiv(W, 128), H, CT);
        upsample_y_kernel<1><<<grid, 128, 0, stream>>>(p, CT, H, W, out_planar);
    }
    OPB_CUDA(cudaGetLastError());
}

// ================================================================================================================
// Batched estimators (srcmx/Batch_model.py Batch_body / Batch_hand, SURVEY.md 8f row N2)
// ================================================================================================================
namespace {

// Front end of Batch_body.__call__ (Batch_model.py:153-155) and Batch_hand.__call__ (:373): float frames in [0,1],
// planar (n,3,H,W); bicubic resize (torch semantics: A = -0.75, half-pixel centres, clamped taps, no antialias) to
// (h,w); minus 0.5; zero padding to (hp,wp).  Output: bf16 HWC3, the input format of conv1_1's bf16 variant.  With
// identical sizes the taps degenerate to (0,1,0,0) and the frame is copied exactly.
// sample (c, y, x) of frame `img`: planar float, or decoded uint8 HWC pixels with ToTensor's division by 255 applied here
__device__ __forceinline__ float frame_at(const float* in, size_t img, int c, int y, int x, int H, int W) {
    return __ldg(in + ((img * 3 + c) * (size_t)H + y) * W + x);
}
__device__ __forceinline__ float frame_at(const uint8_t* in, size_t img, int c, int y, int x, int H, int W) {
    return (float)__ldg(in + ((img * H + y) * (size_t)W + x) * 3 + c) / 255.0f;
}

template <typename TIn>
__global__ void __launch_bounds__(128) preprocess_f32_kernel(const TIn* __restrict__ in, int H, int W,
                                                             __nv_bfloat16* __restrict__ out, int h, int w, int hp, int wp,
                                                             const int* __restrict__ xf, const float* __restrict__ xw,
                                                             const int* __restrict__ yf, const float* __restrict__ yw) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    const size_t img = blockIdx.z;
    if (x >= wp) return;
    float r[3] = {0.f, 0.f, 0.f};
    if (x < w && y < h) {
        const int x0 = xf[x], y0 = yf[y];
        float cx[4], cy[4];
        int xi[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            cx[j] = xw[x * 4 + j];
            cy[j] = yw[y * 4 + j];
            xi[j] = min(max(x0 + j, 0), W - 1);
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            float acc = 0.f;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int yy = min(max(y0 + i, 0), H - 1);
                float t = frame_at(in, img, c, yy, xi[0], H, W) * cx[0];
#pragma unroll
                for (int j = 1; j < 4; ++j) t = t + frame_at(in, img, c, yy, xi[j], H, W) * cx[j];
                acc = acc + t * cy[i];
            }
            r[c] = acc - 0.5f;
        }
    }
    __nv_bfloat16* o = out + ((img * hp + y) * (size_t)wp + x) * 3;
    o[0] = __float2bfloat16_rn(r[0]);
    o[1] = __float2bfloat16_rn(r[1]);
    o[2] = __float2bfloat16_rn(r[2]);
}

}  // namespace

void preprocess_f32_launch(const void* frames, bool frames_u8_hwc, int n, int H, int W, void* out_bf16, int h, int w,
                           int hp, int wp, const int* x_first, const float* x_w, const int* y_first, const float* y_w,
                           cudaStream_t stream) {
    dim3 grid(cdiv(wp, 128), hp, n);
    if (frames_u8_hwc)
        preprocess_f32_kernel<uint8_t><<<grid, 128, 0, stream>>>((const uint8_t*)frames, H, W, (__nv_bfloat16*)out_bf16, h, w,
                                                                 hp, wp, x_first, x_w, y_first, y_w);
    else
        preprocess_f32_kernel<float><<<grid, 128, 0, stream>>>((const float*)frames, H, W, (__nv_bfloat16*)out_bf16, h, w, hp,
                                                               wp, x_first, x_w, y_first, y_w);
    OPB_CUDA(cudaGetLastError());
}

}  // namespace opb
