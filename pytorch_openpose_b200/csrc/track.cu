// Person tracks across frames on the device: the rule of motion.PersonLinker (its docstring is the specification),
// applied to the every-person records of a batch where they already are in device memory.  float64 throughout, every
// product, sum and square root rounded separately (this file is compiled with --fmad=false and uses _rn intrinsics),
// so the ids equal the host linker's bit for bit, float ties included.
//
// One block links the frames of a batch in sequence.  Per frame:
//   drop     tracks that are no longer live, compacted in order (ids stay ascending along the slots);
//   costs    every (live track, person) pair in parallel; the eligible ones appended to a pair list;
//   rank     each pair ranked against the whole list on (cost, track slot, person) -- the keys are unique, so the
//            ranks are a permutation and the order does not depend on the append order or the block size;
//   walk     one thread takes the ranked pairs greedily, as limb_match_kernel does for the limbs;
//   update   matched tracks take the person's body rows, unmatched persons open tracks in person order.
// Track slots are double-buffered: the drop compacts from one buffer into the other.
#include "opb_common.cuh"

namespace opb {
namespace {

constexpr int kTrackThreads = 256;

// exclusive count of the threads before this one (in thread order) whose flag is set, and the block's total; called by
// every thread of the block
__device__ int block_prefix(bool flag, int* s_warp, int& total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned bits = __ballot_sync(0xffffffffu, flag);
    if (lane == 0) s_warp[warp] = __popc(bits);
    __syncthreads();
    int before = 0, all = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
        before += w < warp ? s_warp[w] : 0;
        all += s_warp[w];
    }
    __syncthreads();
    total = all;
    return before + __popc(bits & ((1u << lane) - 1u));
}

// cost of a track (18 x 3 body rows) against a record; false when fewer than min_joints joints are present in both
__device__ __forceinline__ bool pair_cost(const double* __restrict__ t, const double* __restrict__ r, int min_joints,
                                          double& cost) {
    double s = 0.0;
    int n = 0;
    for (int j = 0; j < 18; ++j) {
        if (t[3 * j + 2] > 0.0 && r[3 * j + 2] > 0.0) {
            const double dx = __dsub_rn(r[3 * j], t[3 * j]);
            const double dy = __dsub_rn(r[3 * j + 1], t[3 * j + 1]);
            s = __dadd_rn(s, __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy))));
            ++n;
        }
    }
    if (n < min_joints) return false;
    cost = __ddiv_rn(s, (double)n);
    return true;
}

__device__ __forceinline__ bool pair_before(double c1, int k1, int p1, double c2, int k2, int p2) {
    return c1 < c2 || (c1 == c2 && (k1 < k2 || (k1 == k2 && p1 < p2)));
}

__device__ __forceinline__ void copy_rows(double* __restrict__ dst, const double* __restrict__ src) {
    for (int i = 0; i < 54; ++i) dst[i] = src[i];
}

__global__ void __launch_bounds__(kTrackThreads) track_link_kernel(TrackLink a) {
    __shared__ int s_warp[32];
    __shared__ int s_pairs;
    __shared__ double s_cost[kTrackThreads];
    __shared__ int s_k[kTrackThreads], s_p[kTrackThreads];
    int cur = a.cur, L = a.live, next = a.next_id, g = a.frame;
    size_t rec0 = 0;
    for (int f = 0; f < a.n_frames; ++f, ++g) {
        const int P = a.persons[f];
        const double* rec = a.records + rec0 * 180;
        // drop the tracks that are not live at frame g
        int dead = 0;
        for (int k = threadIdx.x; k < L; k += blockDim.x) dead |= g - a.last[cur][k] > a.max_gap;
        if (__syncthreads_or(dead)) {
            const int nx = cur ^ 1;
            int kept = 0;
            for (int base = 0; base < L; base += blockDim.x) {
                const int k = base + threadIdx.x;
                const bool keep = k < L && g - a.last[cur][k] <= a.max_gap;
                int total;
                const int pos = kept + block_prefix(keep, s_warp, total);
                if (keep) {
                    copy_rows(a.rows[nx] + (size_t)pos * 54, a.rows[cur] + (size_t)k * 54);
                    a.tid[nx][pos] = a.tid[cur][k];
                    a.last[nx][pos] = a.last[cur][k];
                }
                kept += total;
            }
            cur = nx;
            L = kept;
        }
        if (L + P > a.cap || P > a.person_cap) {             // the host sizes the buffers; this cannot happen
            if (threadIdx.x == 0) a.state[4] = 1;
            return;
        }
        // eligible pairs
        if (threadIdx.x == 0) s_pairs = 0;
        __syncthreads();
        const long long LP = (long long)L * P;
        for (long long i = threadIdx.x; i < LP; i += blockDim.x) {
            const int k = (int)(i / P), p = (int)(i % P);
            double c;
            if (pair_cost(a.rows[cur] + (size_t)k * 54, rec + (size_t)p * 180, a.min_joints, c) && c <= a.max_dist) {
                const int e = atomicAdd(&s_pairs, 1);
                if (e < a.pair_cap) {
                    a.pair_cost[e] = c;
                    a.pair_k[e] = k;
                    a.pair_p[e] = p;
                }
            }
        }
        __syncthreads();
        const int E = s_pairs;
        if (E > a.pair_cap) {
            if (threadIdx.x == 0) a.state[4] = 2;
            return;
        }
        // rank every pair against the whole list, one tile of the list in shared memory at a time
        for (int base = 0; base < E; base += blockDim.x) {
            const int e = base + threadIdx.x;
            double c = 0.0;
            int k = 0, p = 0;
            if (e < E) {
                c = a.pair_cost[e];
                k = a.pair_k[e];
                p = a.pair_p[e];
            }
            int rank = 0;
            for (int t0 = 0; t0 < E; t0 += blockDim.x) {
                const int t = t0 + threadIdx.x;
                if (t < E) {
                    s_cost[threadIdx.x] = a.pair_cost[t];
                    s_k[threadIdx.x] = a.pair_k[t];
                    s_p[threadIdx.x] = a.pair_p[t];
                }
                __syncthreads();
                const int m = min((int)blockDim.x, E - t0);
                if (e < E)
                    for (int q = 0; q < m; ++q) rank += pair_before(s_cost[q], s_k[q], s_p[q], c, k, p);
                __syncthreads();
            }
            if (e < E) a.order[rank] = e;
        }
        for (int k = threadIdx.x; k < L; k += blockDim.x) a.track_taken[k] = 0;
        for (int p = threadIdx.x; p < P; p += blockDim.x) a.match[p] = -1;
        __syncthreads();
        // the greedy walk
        if (threadIdx.x == 0) {
            const int limit = min(L, P);
            int count = 0;
            for (int r = 0; r < E && count < limit; ++r) {
                const int e = a.order[r];
                const int k = a.pair_k[e], p = a.pair_p[e];
                if (a.track_taken[k] || a.match[p] >= 0) continue;
                a.track_taken[k] = 1;
                a.match[p] = k;
                ++count;
            }
        }
        __syncthreads();
        // matched tracks take the rows; unmatched persons open tracks, in person order
        int opened = 0;
        for (int base = 0; base < P; base += blockDim.x) {
            const int p = base + threadIdx.x;
            const int k = p < P ? a.match[p] : 0;
            int total;
            const int pos = opened + block_prefix(p < P && k < 0, s_warp, total);
            if (p < P) {
                const int slot = k >= 0 ? k : L + pos;
                if (k < 0) a.tid[cur][slot] = next + pos;
                copy_rows(a.rows[cur] + (size_t)slot * 54, rec + (size_t)p * 180);
                a.last[cur][slot] = g;
                a.ids[rec0 + p] = a.tid[cur][slot];
            }
            opened += total;
        }
        L += opened;
        next += opened;
        rec0 += P;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        a.state[0] = cur;
        a.state[1] = L;
        a.state[2] = next;
        a.state[3] = g;
    }
}

}  // namespace

void track_link_launch(const TrackLink& a, cudaStream_t stream) {
    track_link_kernel<<<1, kTrackThreads, 0, stream>>>(a);
    OPB_CUDA(cudaGetLastError());
}

}  // namespace opb
