// Hand key-point extraction on the device -- src/hand.py:59-75 and util.npmax (src/util.py:205-210).
//
// Per key-point map (21 of the 22 channels) the reference: smooths with gaussian_filter(sigma=3) in float64,
// thresholds at 0.03, labels the binary mask with 8-connectivity, keeps the component with the largest sum of RAW
// map values (first maximum on ties; skimage numbers components in raster order of their first pixel), zeroes
// everything else and takes the first row-major argmax.
//
//   hand_smooth_kernel   same exact-float64 separable filter as peaks.cu; writes label[i] = i for mask pixels,
//                        -1 elsewhere
//   hand_runs / merge / compress / flatten   run-based union-find (atomicMin hooking); roots are the smallest linear
//                        index of a component == raster order of first pixels; per-root float64 sums of raw values
//                        (atomics, in an order that changes from run to run), and per map the mask count M and the
//                        sum A of |value|
//   hand_select_kernel   one CTA per map: the top component by device sum and every component whose device sum is
//                        within the certification bound of it (see select_cut); when another component is that close,
//                        numpy's own sum of each of them (pairwise, in raster order, float64 or float32) decides
//                        (sum desc, root asc); then argmax over pixels of (label == best ? raw : 0) (value desc, index asc)
// The choice of component therefore equals the reference's whatever order the atomics ran in.
#include "opb_common.cuh"

#include <algorithm>
#include <climits>
#include <mutex>

namespace opb {
namespace {

constexpr int TW = 32, TH = 16, R = kGaussRadius;
constexpr int RAW_W = TW + 2 * R, RAW_H = TH + 2 * R;

__device__ __forceinline__ int reflect_idx(int i, int n) {
    const int period = 2 * n;
    i %= period;
    if (i < 0) i += period;
    return i >= n ? period - 1 - i : i;
}

// Ragged batches (crops of different sizes in one launch, the per-frame caller's hand boxes): `dims` holds the side
// length of every (square) crop, the planes of a crop are stored densely with that width at a fixed stride `ps`, and
// the grids are sized for the largest crop; dims == null means one size (h, w) for all, ps = h * w.
#define OPB_HAND_GEOM(crop)                  \
    if (dims) {                              \
        h = w = dims[crop];                  \
    }

__global__ void __launch_bounds__(256) hand_smooth_kernel(const float* __restrict__ heat, int h, int w, int chan_stride_maps,
                                                          const GaussTaps taps, double thre, int* __restrict__ labels,
                                                          double* __restrict__ smoothed_out, const int* __restrict__ dims,
                                                          size_t ps, double* __restrict__ sums, double* __restrict__ mask_acc) {
    __shared__ double raw[RAW_H][RAW_W];
    __shared__ double ver[TH][RAW_W];
    const int m = blockIdx.z;                                   // map index = crop * 21 + part
    const int crop = m / 21, part = m - crop * 21;
    OPB_HAND_GEOM(crop)
    const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH;
    if (x0 >= w || y0 >= h) return;
    const float* map = heat + ((size_t)crop * chan_stride_maps + part) * ps;
    const int tid = threadIdx.x;
    if (x0 == 0 && y0 == 0 && tid < 2) mask_acc[(size_t)m * 3 + tid] = 0.0;     // A and M of this map (hand_flatten_kernel)
    __shared__ int s_row[RAW_H], s_col[RAW_W];
    if (tid < RAW_H) s_row[tid] = reflect_idx(y0 - R + tid, h);
    else if (tid < RAW_H + RAW_W) s_col[tid - RAW_H] = reflect_idx(x0 - R + (tid - RAW_H), w);
    __syncthreads();
    {
        constexpr int PER = (RAW_H * RAW_W + 255) / 256;       // batch the halo loads (memory-level parallelism)
        float vals[PER];
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            const int i = tid + j * 256;
            const int ry = i / RAW_W, rx = i - ry * RAW_W;
            vals[j] = i < RAW_H * RAW_W ? __ldg(map + (size_t)s_row[ry] * w + s_col[rx]) : 0.f;
        }
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            const int i = tid + j * 256;
            if (i < RAW_H * RAW_W) raw[i / RAW_W][i % RAW_W] = (double)vals[j];
        }
    }
    __syncthreads();
    for (int i = tid; i < TH * RAW_W; i += blockDim.x) {
        const int r = i / RAW_W, c = i - r * RAW_W;
        double acc = __dmul_rn(raw[r + R][c], taps.w[0]);
#pragma unroll
        for (int d = R; d >= 1; --d)
            acc = __dadd_rn(acc, __dmul_rn(__dadd_rn(raw[r + R - d][c], raw[r + R + d][c]), taps.w[d]));
        ver[r][c] = acc;
    }
    __syncthreads();
    for (int i = tid; i < TH * TW; i += blockDim.x) {
        const int ty = i / TW, tx = i - ty * TW;
        const int y = y0 + ty, x = x0 + tx;
        if (y >= h || x >= w) continue;
        double acc = __dmul_rn(ver[ty][tx + R], taps.w[0]);
#pragma unroll
        for (int d = R; d >= 1; --d)
            acc = __dadd_rn(acc, __dmul_rn(__dadd_rn(ver[ty][tx + R - d], ver[ty][tx + R + d]), taps.w[d]));
        const size_t idx = (size_t)m * ps + (size_t)y * w + x;
        labels[idx] = acc > thre ? y * w + x : -1;
        sums[idx] = 0.0;                                        // per-root sums are accumulated by hand_flatten_kernel
        if (smoothed_out) smoothed_out[idx] = acc;
    }
}

// parent reads go to L2 (__ldcg): other CTAs hook roots with atomics while we walk
__device__ __forceinline__ int uf_find(const int* L, int x) {
    int p = __ldcg(L + x);
    while (p != x) {
        x = p;
        p = __ldcg(L + x);
    }
    return x;
}
__device__ void uf_union(int* L, int a, int b) {
    while (true) {
        a = uf_find(L, a);
        b = uf_find(L, b);
        if (a == b) return;
        if (a > b) {
            const int t = a;
            a = b;
            b = t;
        }
        const int old = atomicMin(&L[b], a);        // hook the larger root under the smaller
        if (old == b) return;
        b = old;
    }
}

// ---- connected components, 8-connectivity -------------------------------------------------------------------------
// Labels are built run-first so that even one giant component (a map that is above the threshold everywhere) stays
// cheap: (1) every mask pixel points at the first pixel of its horizontal run, (2) runs of adjacent rows are united
// once per touching pair (union-find over run heads only, atomicMin hooking: the root is the smallest raster index
// of the component), (3) run heads are compressed to their root, (4) every pixel resolves label[label[i]].

// (1) one warp per image row
__global__ void hand_runs_kernel(int* __restrict__ labels, int h, int w, const int* __restrict__ dims, size_t ps) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    OPB_HAND_GEOM(blockIdx.y / 21)
    if (row >= h) return;
    int* L = labels + (size_t)blockIdx.y * ps + (size_t)row * w;
    int carry = -1;                                     // head of the run that reaches the start of this segment
    for (int x0 = 0; x0 < w; x0 += 32) {
        const int x = x0 + lane;
        const bool on = x < w && L[x] >= 0;
        const unsigned bits = __ballot_sync(0xffffffffu, on);
        // closest zero bit strictly below this lane
        const unsigned below = ~bits & ((1u << lane) - 1);
        int head;
        if (below) head = x0 + (32 - __clz(below));     // run starts right after the highest zero below
        else head = carry >= 0 ? carry : x0;            // run reaches the segment start
        if (on) L[x] = row * w + head;
        // carry for the next segment: head of the run containing lane 31, if any
        const int head31 = __shfl_sync(0xffffffffu, head, 31);
        carry = (bits >> 31) ? head31 : -1;
    }
}

// (2) unite every run with the runs of the row above that touch it (columns xs-1 .. xe+1)
constexpr int kRowsPerBlock = 16;     // rows a block of the per-pixel passes walks (ragged batches size their grids for the largest crop)
__global__ void hand_merge_kernel(int* __restrict__ labels, int h, int w, const int* __restrict__ dims, size_t ps) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    OPB_HAND_GEOM(blockIdx.z / 21)
    if (x >= w) return;
    int* L = labels + (size_t)blockIdx.z * ps;
    for (int y = max(1, (int)blockIdx.y * kRowsPerBlock); y < min(h, ((int)blockIdx.y + 1) * kRowsPerBlock); ++y) {
        const int i = y * w + x;
        const int mine = L[i];
        if (mine < 0) continue;
        const int* up = L + i - w;
        const bool u0 = up[0] >= 0;
        // an upper run that STARTS at x+1 touches this run
        if (x + 1 < w && up[1] >= 0 && !u0) uf_union(L, mine, up[1]);
        // at the head of this run (decided by geometry: the head's own entry may already have been hooked by another
        // thread): the upper run covering x-1 or x
        if (x == 0 || L[i - 1] < 0) {
            if (x > 0 && up[-1] >= 0) uf_union(L, mine, up[-1]);
            else if (u0) uf_union(L, mine, up[0]);
        }
    }
}

// (3) compress run heads to their roots
__global__ void hand_compress_kernel(int* __restrict__ labels, int h, int w, const int* __restrict__ dims, size_t ps) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    OPB_HAND_GEOM(blockIdx.z / 21)
    if (x >= w) return;
    int* L = labels + (size_t)blockIdx.z * ps;
    for (int y = blockIdx.y * kRowsPerBlock; y < min(h, ((int)blockIdx.y + 1) * kRowsPerBlock); ++y) {
        const int i = y * w + x;
        if (L[i] < 0) continue;
        const bool head = x == 0 || L[i - 1] < 0;
        if (!head) continue;
        const int root = uf_find(L, i);
        if (root != i) L[i] = root;                        // only ever lowers an entry towards its root
    }
}

// (4) resolve every pixel and accumulate the raw-map sum of its component; per map, the mask count M and the sum A of
// |value| (mask_acc[m * 3 + 1] and mask_acc[m * 3 + 0]) for the certification bound of hand_select_kernel
__global__ void hand_flatten_kernel(const float* __restrict__ heat, int chan_stride_maps, int* __restrict__ labels,
                                    double* __restrict__ sums, int h, int w, const int* __restrict__ dims, size_t ps,
                                    double* __restrict__ mask_acc) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int m = blockIdx.z;
    const int crop = m / 21, part = m - crop * 21;
    OPB_HAND_GEOM(crop)
    int* L = labels + (size_t)m * ps;
    if ((int)(blockIdx.x * blockDim.x) >= w) return;
    int count = 0;
    double absum = 0.0;
    for (int y = blockIdx.y * kRowsPerBlock; y < min(h, ((int)blockIdx.y + 1) * kRowsPerBlock); ++y) {
        const int i = y * w + x;
        int root = -1;
        double v = 0.0;
        if (x < w && L[i] >= 0) {
            root = __ldcg(L + __ldcg(L + i));              // pixel -> run head -> root
            // a run head may itself still point one hop short if it was hooked after its own compression pass started
            root = uf_find(L, root);
            L[i] = root;
            v = (double)heat[((size_t)crop * chan_stride_maps + part) * ps + i];
            count += 1;
            absum += fabs(v);
        }
        // warp-aggregated atomics: lanes of a warp almost always share one root
        const unsigned active = __ballot_sync(0xffffffffu, root >= 0);
        if (root < 0) continue;
        const unsigned same = __match_any_sync(active, root);
        if (active == 0xffffffffu && same == active) {
            double tot = v;
#pragma unroll
            for (int o = 16; o; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
            if ((threadIdx.x & 31) == 0) atomicAdd(&sums[(size_t)m * ps + root], tot);
        } else {
            atomicAdd(&sums[(size_t)m * ps + root], v);
        }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        count += __shfl_xor_sync(0xffffffffu, count, o);
        absum += __shfl_xor_sync(0xffffffffu, absum, o);
    }
    if ((threadIdx.x & 31) == 0 && count) {
        atomicAdd(&mask_acc[(size_t)m * 3 + 0], absum);
        atomicAdd(&mask_acc[(size_t)m * 3 + 1], (double)count);
    }
}

struct Best {
    double v;
    int idx;
};
__device__ __forceinline__ Best better(Best a, Best b) {       // value descending, index ascending
    if (b.idx >= 0 && (a.idx < 0 || b.v > a.v || (b.v == a.v && b.idx < a.idx))) return b;
    return a;
}
__device__ Best block_best(Best mine, Best* s) {
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        Best other;
        other.v = __shfl_xor_sync(0xffffffffu, mine.v, o);
        other.idx = __shfl_xor_sync(0xffffffffu, mine.idx, o);
        mine = better(mine, other);
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncthreads();
    if (lane == 0) s[warp] = mine;
    __syncthreads();
    Best r = s[0];
    for (int i = 1; i < (int)(blockDim.x >> 5); ++i) r = better(r, s[i]);
    return r;
}

// the best component and the runner-up
struct Top2 {
    Best a, b;
};
__device__ __forceinline__ Top2 top2_merge(Top2 x, Top2 y) {
    Top2 r;
    r.a = better(x.a, y.a);
    const Best other = r.a.idx == x.a.idx ? y.a : x.a;       // valid indices are distinct
    r.b = better(better(x.b, y.b), other);
    return r;
}
__device__ Top2 block_top2(Top2 mine, Top2* s) {
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        Top2 other;
        other.a.v = __shfl_xor_sync(0xffffffffu, mine.a.v, o);
        other.a.idx = __shfl_xor_sync(0xffffffffu, mine.a.idx, o);
        other.b.v = __shfl_xor_sync(0xffffffffu, mine.b.v, o);
        other.b.idx = __shfl_xor_sync(0xffffffffu, mine.b.idx, o);
        mine = top2_merge(mine, other);
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncthreads();
    if (lane == 0) s[warp] = mine;
    __syncthreads();
    Top2 r = s[0];
    for (int i = 1; i < (int)(blockDim.x >> 5); ++i) r = top2_merge(r, s[i]);
    return r;
}

// γ_k = k·u / (1 − k·u), rounded up
__device__ __forceinline__ double gamma_ru(double k, double u) {
    const double ku = k * u;                                     // exact: k an integer < 2^53, u a power of two
    return __ddiv_ru(ku, __dadd_rd(1.0, -ku));
}

// Certification bound.  Every component c of a map has m_c <= M values with sum of magnitudes A_c <= A (M and A of the
// whole mask, from hand_flatten_kernel).  Any float64 summation order of m values -- the device's warp trees and atomics
// as well as numpy's pairwise order -- is within γ_(m-1)·Σ|v| of the exact sum (Higham, Accuracy and Stability of
// Numerical Algorithms, §4.2), with u = 2^-53.  numpy's float32 pairwise sum (Batch_hand) is within γ_d·Σ|v| with
// u = 2^-24, d the largest number of roundings one element passes through in pairwise_block (pairwise_depth_max, taken
// over every length up to the map's pixel count, so it covers any component).  So for every component
//     |S_dev − S_numpy| <= B = (γ_M(2^-53) + γ')·A,   γ' = γ_M(2^-53) (Hand) or γ_d(2^-24) (Batch_hand).
// A itself is a float64 sum of M magnitudes: A >= A_true·(1 − γ_M), so A_true <= A / (1 − γ_M).  If w is the
// reference's winner and t the device's top component, S_dev(w) >= S_np(w) − B >= S_np(t) − B >= S_dev(t) − 2B: every
// component with S_dev >= S_dev(t) − 2B is a contender, the reference's winner among them.  All of it rounds outwards.
__device__ double select_cut(double top, double A, double M, int f32_depth) {
    const double g = gamma_ru(M, 0x1p-53);
    const double a_up = __ddiv_ru(A, __dadd_rd(1.0, -M * 0x1p-53));
    const double g2 = f32_depth ? gamma_ru((double)f32_depth, 0x1p-24) : g;
    const double bound = __dmul_ru(__dadd_ru(g, g2), a_up);
    return __dadd_rd(top, -__dmul_ru(2.0, bound));
}

// numpy_sum of buf[0, n) by the whole CTA: thread t evaluates the subtree of pairwise_block reached by following the
// ten bits of t from the top (a node that is already a leaf above that depth belongs to the thread whose remaining bits
// are 0); thread 0 then adds the partial sums up the same tree.  The result is numpy_sum's, bit for bit.
// The walk of pairwise_block over the top ten levels, with part[t] at the nodes there: level k of the path is bit
// 9 - k of t.
template <typename T>
__device__ T subtree_combine(long long n, const T* part) {
    T left[10];
    long long right[10];
    unsigned has_left = 0;
    int sp = 0, t = 0;
    long long len = n;
    while (true) {
        while (sp < 10 && len > 128) {
            const long long n2 = pairwise_split(len);
            right[sp] = len - n2;
            has_left &= ~(1u << sp);
            ++sp;
            len = n2;
        }
        T val = part[t];
        while (sp > 0 && (has_left >> (sp - 1) & 1)) {
            --sp;
            val = left[sp] + val;
            t &= ~(1 << (9 - sp));
        }
        if (sp == 0) return val;
        left[sp - 1] = val;
        has_left |= 1u << (sp - 1);
        len = right[sp - 1];
        t |= 1 << (9 - (sp - 1));
    }
}
template <typename T>
__device__ T block_numpy_sum(const T* buf, long long n, T* part) {
    const int t = threadIdx.x;
    long long off = 0, len = n;
    bool own = true;
    for (int lv = 9; lv >= 0; --lv) {
        const bool right = (t >> lv) & 1;
        if (len > 128) {
            const long long n2 = pairwise_split(len);
            if (right) off += n2, len -= n2;
            else len = n2;
        } else if (right) {
            own = false;
        }
    }
    if (own) part[t] = pairwise_block(buf + off, len);
    __syncthreads();
    if (t == 0) part[0] = T(0) + subtree_combine(n, part);
    __syncthreads();
    const T r = part[0];
    __syncthreads();                                             // part is reused by the next call
    return r;
}

// The exact path of hand_select_kernel: numpy's sum of every contender (root r with S[r] >= cut), the best of them
// (sum desc, root asc).  Contender roots are marked in the label plane (L[r] = -2 - r) and restored one by one; the
// device sums are not needed once they are marked, so component r's values are compacted in raster order into the
// sums plane from index r on (its pixels all lie at r or later, so they fit) and its exact sum is left at S[r], where
// no later contender's compaction reaches.  O(map) per contender.
template <typename T>
__device__ __noinline__ Best exact_choice(const float* map, int* L, double* S, int n, double cut) {
    __shared__ T part[1024];
    __shared__ int wcnt[2][32];
    __shared__ int s_min[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    for (int i = tid; i < n; i += blockDim.x)
        if (L[i] == i && S[i] >= cut) L[i] = -2 - i;
    __syncthreads();
    Best win{0.0, -1};
    int r = -1;
    int par = 0;
    while (true) {
        int first = INT_MAX;                                     // next contender: the smallest marked root
        for (int i = r + 1 + tid; i < n; i += blockDim.x)
            if (L[i] <= -2) {
                first = i;
                break;
            }
#pragma unroll
        for (int o = 16; o; o >>= 1) first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
        if (lane == 0) s_min[warp] = first;
        __syncthreads();
        r = INT_MAX;
        for (int k = 0; k < nwarps; ++k) r = min(r, s_min[k]);
        __syncthreads();
        if (r == INT_MAX) break;
        T* buf = reinterpret_cast<T*>(S + r);
        long long cnt = 0;
        for (int i0 = r; i0 < n; i0 += blockDim.x) {
            const int i = i0 + tid;
            const bool on = i < n && (i == r || L[i] == r);
            const unsigned bal = __ballot_sync(0xffffffffu, on);
            if (lane == 0) wcnt[par][warp] = __popc(bal);
            __syncthreads();
            int pre = 0, tot = 0;
            for (int k = 0; k < nwarps; ++k) {
                const int c = wcnt[par][k];
                pre += k < warp ? c : 0;
                tot += c;
            }
            if (on) buf[cnt + pre + __popc(bal & ((1u << lane) - 1))] = (T)map[i];
            cnt += tot;
            par ^= 1;
        }
        __syncthreads();
        const T sum = block_numpy_sum(buf, cnt, part);
        if (tid == 0) {
            S[r] = (double)sum;
            L[r] = r;
        }
        win = better(win, Best{(double)sum, r});
        __syncthreads();
    }
    return win;
}

__global__ void __launch_bounds__(1024, 2) hand_select_kernel(const float* __restrict__ heat, int chan_stride_maps,
                                                           int* labels, double* sums, int h, int w,
                                                           double* __restrict__ peaks, const int* __restrict__ dims,
                                                           size_t ps, int f32_depth, bool exact_all) {
    __shared__ Best s[32];
    __shared__ Top2 s2[32];
    const int m = blockIdx.x;
    const int crop = m / 21, part = m - crop * 21;
    OPB_HAND_GEOM(crop)
    const int n = h * w;
    int* L = labels + (size_t)m * ps;
    double* S = sums + (size_t)m * ps;
    const float* map = heat + ((size_t)crop * chan_stride_maps + part) * ps;
    const double A = peaks[(size_t)m * 3 + 0], M = peaks[(size_t)m * 3 + 1];   // read before anything writes peaks
    Top2 mine2{{0.0, -1}, {0.0, -1}};
    for (int i = threadIdx.x; i < n; i += blockDim.x)
        if (L[i] == i) mine2 = top2_merge(mine2, Top2{{S[i], i}, {0.0, -1}});     // roots only
    const Top2 top = block_top2(mine2, s2);
    Best comp = top.a;
    if (comp.idx < 0) {                                          // nothing above the threshold: [0, 0, 0]
        if (threadIdx.x < 3) peaks[(size_t)m * 3 + threadIdx.x] = 0.0;
        return;
    }
    const double cut = exact_all ? -INFINITY : select_cut(comp.v, A, M, f32_depth);
    if (exact_all || (top.b.idx >= 0 && top.b.v >= cut))
        comp = f32_depth ? exact_choice<float>(map, L, S, n, cut) : exact_choice<double>(map, L, S, n, cut);
    Best mine{0.0, -1};
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double v = L[i] == comp.idx ? (double)map[i] : 0.0;   // map_ori[label_img == 0] = 0
        mine = better(mine, Best{v, i});
    }
    const Best px = block_best(mine, s);
    if (threadIdx.x == 0) {
        peaks[(size_t)m * 3 + 0] = (double)(px.idx % w);
        peaks[(size_t)m * 3 + 1] = (double)(px.idx / w);
        peaks[(size_t)m * 3 + 2] = px.v;
    }
}

// Batch_hand (srcmx/Batch_model.py:391-392): the map is already blurred; mask = value > thre, compared in float32
__global__ void hand_mask_kernel(const float* __restrict__ heat, int h, int w, int chan_stride_maps, float thre,
                                 int* __restrict__ labels, double* __restrict__ sums, double* __restrict__ mask_acc) {
    const int m = blockIdx.z;
    const int crop = m / 21, part = m - crop * 21;
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (blockIdx.x == 0 && y == 0 && threadIdx.x < 2) mask_acc[(size_t)m * 3 + threadIdx.x] = 0.0;   // A and M (flatten)
    if (x >= w) return;
    const float v = __ldg(heat + ((size_t)crop * chan_stride_maps + part) * h * w + (size_t)y * w + x);
    labels[(size_t)m * h * w + (size_t)y * w + x] = v > thre ? y * w + x : -1;
    sums[(size_t)m * h * w + (size_t)y * w + x] = 0.0;
}

}  // namespace

static void hand_components_launch(const float* heat_planar, int maps, int chan_stride_maps, int h, int w, HandBuffers hb,
                                   const int* dims, size_t ps, int f32_depth, cudaStream_t stream);

// The most roundings one element passes through in pairwise_block over n values (n < 8: r = 0 + a[0] + ...; up to 128:
// its accumulator, the three-level tree, the n % 8 tail; above: one more per split) ...
static int pairwise_depth(const std::vector<unsigned char>& d, long long n) {
    if (n < 8) return (int)n;
    if (n <= 128) return (int)(n / 8 - 1 + 3 + n % 8);
    const long long n2 = pairwise_split(n);
    return 1 + std::max(d[n2], d[n - n2]);
}
// ... and its maximum over every length up to n, the float32 error order of numpy's sum of any component of a map of n
// pixels.  Tabulated once per process up to the largest n asked for (a byte per length).
static int pairwise_depth_max(long long n) {
    static std::mutex mu;
    static std::vector<unsigned char> d{0}, dmax{0};
    std::lock_guard<std::mutex> lock(mu);
    for (long long k = (long long)d.size(); k <= n; ++k) {
        d.push_back((unsigned char)pairwise_depth(d, k));
        dmax.push_back(std::max(dmax.back(), d.back()));
    }
    return dmax[n];
}

// Batch_hand post-processing (srcmx/Batch_model.py:387-406): threshold, component sums and the maximum all on the
// blurred map that is passed in.
void hand_peaks_blurred_launch(const float* blurred_planar, int n_crops, int chan_stride_maps, int h, int w, float thre,
                               HandBuffers hb, cudaStream_t stream) {
    const int maps = n_crops * 21;
    OPB_REQUIRE(maps <= 65535, "hand_peaks: too many crops in one batch");
    dim3 g(cdiv(w, 128), h, maps);
    hand_mask_kernel<<<g, 128, 0, stream>>>(blurred_planar, h, w, chan_stride_maps, thre, hb.labels, hb.sums, hb.peaks);
    OPB_CUDA(cudaGetLastError());
    hand_components_launch(blurred_planar, maps, chan_stride_maps, h, w, hb, nullptr, (size_t)h * w,
                           pairwise_depth_max((long long)h * w), stream);
}

// heat: planar (n_crops * chan_stride_maps, h, w) fp32, the first 21 planes of each crop are used
void hand_peaks_launch2(const float* heat_planar, int n_crops, int chan_stride_maps, int h, int w, double thre,
                        HandBuffers hb, double* smoothed_out, cudaStream_t stream) {
    const int maps = n_crops * 21;
    OPB_REQUIRE(maps <= 65535, "hand_peaks: too many crops in one batch");
    dim3 g1(cdiv(w, TW), cdiv(h, TH), maps);
    hand_smooth_kernel<<<g1, 256, 0, stream>>>(heat_planar, h, w, chan_stride_maps, gauss_taps_sigma3(), thre,
                                               hb.labels, smoothed_out, nullptr, (size_t)h * w, hb.sums, hb.peaks);
    OPB_CUDA(cudaGetLastError());
    hand_components_launch(heat_planar, maps, chan_stride_maps, h, w, hb, nullptr, (size_t)h * w, 0, stream);
}

// ragged batch: crop c is dims[c] x dims[c] (0: no crop, peaks are zero), planes at stride wmax * wmax
void hand_peaks_ragged_launch(const float* heat_planar, int n_crops, int chan_stride_maps, const int* dims_dev, int wmax,
                              double thre, HandBuffers hb, cudaStream_t stream) {
    const int maps = n_crops * 21;
    OPB_REQUIRE(maps <= 65535, "hand_peaks: too many crops in one batch");
    const size_t ps = (size_t)wmax * wmax;
    dim3 g1(cdiv(wmax, TW), cdiv(wmax, TH), maps);
    hand_smooth_kernel<<<g1, 256, 0, stream>>>(heat_planar, wmax, wmax, chan_stride_maps, gauss_taps_sigma3(), thre,
                                               hb.labels, nullptr, dims_dev, ps, hb.sums, hb.peaks);
    OPB_CUDA(cudaGetLastError());
    hand_components_launch(heat_planar, maps, chan_stride_maps, wmax, wmax, hb, dims_dev, ps, 0, stream);
}

// labels hold the mask (own raster index or -1): components, per-component sums, selection (src/hand.py:68-74);
// f32_depth: 0 = numpy sums in float64 (Hand), else pairwise_depth_max of the map size (Batch_hand's float32 sums)
static void hand_components_launch(const float* heat_planar, int maps, int chan_stride_maps, int h, int w, HandBuffers hb,
                                   const int* dims, size_t ps, int f32_depth, cudaStream_t stream) {
    dim3 g2(cdiv(w, 128), cdiv(h, kRowsPerBlock), maps);
    dim3 g0(cdiv(h, 4), maps);
    hand_runs_kernel<<<g0, 128, 0, stream>>>(hb.labels, h, w, dims, ps);
    OPB_CUDA(cudaGetLastError());
    hand_merge_kernel<<<g2, 128, 0, stream>>>(hb.labels, h, w, dims, ps);
    OPB_CUDA(cudaGetLastError());
    hand_compress_kernel<<<g2, 128, 0, stream>>>(hb.labels, h, w, dims, ps);
    OPB_CUDA(cudaGetLastError());
    hand_flatten_kernel<<<g2, 128, 0, stream>>>(heat_planar, chan_stride_maps, hb.labels, hb.sums, h, w, dims, ps, hb.peaks);
    OPB_CUDA(cudaGetLastError());
    hand_select_kernel<<<maps, 1024, 0, stream>>>(heat_planar, chan_stride_maps, hb.labels, hb.sums, h, w, hb.peaks, dims, ps,
                                                  f32_depth, hb.exact_all);
    OPB_CUDA(cudaGetLastError());
}

}  // namespace opb
