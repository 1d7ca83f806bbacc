// CTA-pair (tcgen05 cta_group::2) variant of the patch-resident convolution (conv_patch.cu, MODE 1).
//
// Why: with cta_group::1 every 128x128x16 UMMA reads 4 KB of A and 4 KB of B from shared memory in 64 cycles
// (128 B/clk) while TMA keeps writing ~45 B/clk into the same shared memory; ncu shows the tensor pipe 82 % busy.
// A CTA pair issues ONE UMMA with M = 256: each SM contributes its own 128 A rows (its own halo patch, its own
// TMEM accumulator) and only HALF of the weight tile (N/2 rows), so per SM the operand reads drop to 6 KB per 64
// cycles and the weight traffic L2->SM halves.
//
//   cluster (2,1,1): CTA rank r owns super-tile 2*pair + r of a problem (same weights, same n tile, same orientation).
//   leader (rank 0) : arms the full barriers for the bytes of BOTH CTAs, issues every tcgen05.mma.cta_group::2 -- two
//                     issuer warps, one per 128-pixel half of the super-tiles -- and commits with .multicast::cluster so
//                     the empty / accumulator-full barriers of both CTAs fire (two arrivals each, one per issuer).
//   both CTAs       : TMA producers (patches + their half of the weights; complete_tx goes to the leader's barrier),
//                     epilogue (own TMEM rows), which releases the accumulator by arriving on the LEADER's barrier.
//   8 warps         : 0 weight producer, 1 and 7 MMA issuers (1 also owns the TMEM allocation), 2-5 epilogue, 6 patch producer.
//
// Per-launch variations, all decided on the host (conv_pair_plan): tile classes and orientations (QProb), 16 x 8 tiles and
// a 64-wide N tile for launches that fill few SMs, K chunks that are skipped or multiplied at half the N extent (the
// wide-pixel form of conv1_2, net.cu), a weight set that stays in shared memory for the whole kernel (bres).
#include "opb_common.cuh"
#include "tc_ptx.cuh"
#include <cstdlib>
#include <algorithm>

namespace opb {
namespace {

using namespace tc;

constexpr int kThreads = 256;
constexpr int kAccStages = 2;
constexpr int kHalves = 2;
constexpr int kTile = 16;
constexpr int kPitch = 16;
constexpr int FLAG_RELU = 1, FLAG_F32 = 2, FLAG_POOL = 4, FLAG_POOLW = 8;

struct QProb {
    void* out;
    const float* bias;
    int H, W, N;
    int tiles_x, tiles_y;
    int m_tiles, m_pairs;        // super-tiles of the problem, and pairs of them (rounded up)
    int out_cstride, cout_store;
    int n_tiles_n, cin_chunks;
    int pair_begin, flags;       // pair_begin: first index of the problem's full-cost pairs in the launch's pair order
    int edge_begin;              // first index of its half-cost pairs (both tiles have an empty half), after ALL full-cost pairs
    int n_full_pairs;            // pairs of the problem whose first tile has two occupied halves (x n_tiles_n in the order)
    int tile_h;                  // 16, or 8 for small problems: one 16 x 8 half per CTA, twice the CTA pairs, half the K-loop depth
    int noskip;                  // A/B switch: multiply empty halves too
    int vsplit;                  // orientation of the tiles with two occupied halves: 0 = the two 128-pixel halves sit side by
                                 // side (8 cols x 16 rows each), 1 = stacked (16 cols x 8 rows each)
    // Tile classes (in this order in the problem's tile list, each padded to an even count so that the two tiles of a CTA
    // pair always share class and orientation):  F = both halves hold pixels (fx x fy tiles per image);  C = last tile
    // column when at most 8 image columns remain there: side by side, left half only (fy per image);  R = last tile row
    // when at most 8 rows remain: stacked, top half only (tiles_x per image, corner included).
    int fx, fy;
    int nF, nC, nR;              // real tiles per class over all images
    int startC, startR;          // first tile index of class C / R (even)
};

struct alignas(64) PairParams {
    CUtensorMap tmA[kConvMaxProblems];
    CUtensorMap tmW[kConvMaxProblems];
    QProb prob[kConvMaxProblems];
    int nprob, total_pairs, ks;
    int total_full;              // pairs [0, total_full) are full-cost, [total_full, total_pairs) half-cost: the round robin over
                                 // CTA pairs then gives every cluster the same share of each, and the last round is a cheap one
    CUtensorMap tmWh;            // the weights of problem 0 with a box of a quarter N tile (half chunks; all problems share them)
    unsigned khalf_lo, khalf_hi; // bit (chunk * ks + dx): only the lower / upper half of the N tile has non-zero weights there
    int n_patch;                 // patch buffers in flight (4 for 3x3 layers, 3 for 7x7)
    int bres;                    // > 0: one weight set of one N tile whose chunks all fit the weight stages (conv1_2 wide form, conv2_1):
                                 // loaded once per CTA (bres bytes), never recycled
    unsigned kskip;              // bit (chunk * ks + dx): that 64-channel chunk of column tap dx has all-zero weights (ConvOp::kskip)
    int resident;                // short-K layers (conv1_2: 3x3, 64 channels, one weight set): the 9 weight taps stay in shared
                                 // memory for the whole kernel and ONE 24-column patch per tile serves all three dx
};
static_assert(sizeof(PairParams) <= 4000, "kernel parameter space");

template <int BLOCK_N>
struct QCfg {
    static constexpr int kPatchBytesMax = kPitch * (kTile + 6) * 128;      // 45056 (ks = 7)
    static constexpr int kNumPatch = 4;                                    // barriers; ks = 7 uses three buffers (n_patch below)
    static constexpr int kPatchBytes3 = kPitch * (kTile + 2) * 128;        // 36864 (ks = 3): four of them
    static constexpr int kPatchRegion = 4 * kPatchBytes3 > 3 * kPatchBytesMax ? 4 * kPatchBytes3 : 3 * kPatchBytesMax;
    static constexpr int kBHalfBytes = (BLOCK_N / 2) * 128;                 // this CTA's half of a weight stage
    static constexpr int kBStages = 9;       // 9: room for every weight chunk of a short-K layer (bres / resident modes)
    static constexpr int kResPitch = 24;                                   // resident mode: patch columns (18 used)
    static constexpr int kResPatchBytes = kResPitch * (kTile + 2) * 128;   // 55296
    static constexpr int kResPatchStride = (kPatchRegion / 2) / 1024 * 1024;   // two buffers in the patch region
    static_assert(kResPatchBytes <= kResPatchStride, "resident patch buffers");
    static constexpr int kTmemCols = kAccStages * kHalves * BLOCK_N;
    static constexpr int kNumBars = 2 * kNumPatch + 2 * kBStages + 2 * kAccStages;
    static constexpr int kBarBytes = kNumBars * 8 + 16;
    static constexpr int kBiasBytes = kAccStages * BLOCK_N * 4;
    static constexpr int kSmemBytes = 1024 + kPatchRegion + kBStages * kBHalfBytes + kBarBytes + kBiasBytes;
    static_assert(kBHalfBytes % 1024 == 0, "swizzle atoms must stay 1024-B aligned");
    static_assert(kSmemBytes <= 232448, "shared memory budget");
};

__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(sbo_bytes >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

// mask bit of K chunk `i` = channel chunk * ks + dx (layers with more than 32 chunks have no masks)
__host__ __device__ __forceinline__ unsigned chunk_bit(int i) { return i < 32 ? 1u << i : 0u; }

struct TileCoord {
    int pi, img, x0, y0, n0;
    bool real;                   // false: padding tile of an odd problem (computed, never stored)
    int halves;                  // bit h: half h of the super-tile holds at least one pixel of the image
    int vsplit;                  // orientation of this tile (QProb::vsplit for class F, 0 for C, 1 for R)
};
__host__ __device__ __forceinline__ TileCoord decode_pair(const PairParams& p, int pr, int rank, int block_n) {
    int pi = 0, local;
    if (pr < p.total_full) {
        while (pi + 1 < p.nprob && pr >= p.prob[pi + 1].pair_begin) ++pi;
        local = pr - p.prob[pi].pair_begin;
    } else {
        while (pi + 1 < p.nprob && pr >= p.prob[pi + 1].edge_begin) ++pi;
        local = pr - p.prob[pi].edge_begin + p.prob[pi].n_full_pairs * p.prob[pi].n_tiles_n;
    }
    const QProb& q = p.prob[pi];
    const int nt = local % q.n_tiles_n;
    const int mp = local / q.n_tiles_n;
    const int mt = 2 * mp + rank;
    TileCoord c;
    int img, txi, tyi, idx;
    if (mt < q.startC) {                                  // class F, row-major inside an image
        idx = mt;
        c.real = idx < q.nF;
        if (!c.real) idx = q.nF - 1;
        const int per = q.fx * q.fy;
        img = idx / per;
        const int r = idx - img * per;
        tyi = r / q.fx;
        txi = r - tyi * q.fx;
        c.vsplit = q.vsplit;
        c.halves = (q.tile_h == kTile) ? 3 : 1;
    } else if (mt < q.startR) {                           // class C
        idx = mt - q.startC;
        c.real = idx < q.nC;
        if (!c.real) idx = q.nC - 1;
        img = idx / q.fy;
        tyi = idx - img * q.fy;
        txi = q.tiles_x - 1;
        c.vsplit = 0;
        c.halves = 1;
    } else {                                              // class R
        idx = mt - q.startR;
        c.real = idx < q.nR;
        if (!c.real) idx = q.nR - 1;
        img = idx / q.tiles_x;
        txi = idx - img * q.tiles_x;
        tyi = q.tiles_y - 1;
        c.vsplit = 1;
        c.halves = 1;
    }
    c.pi = pi;
    c.img = img;
    c.x0 = txi * kTile;
    c.y0 = tyi * q.tile_h;
    c.n0 = nt * block_n;
    if (!c.real) c.halves = 0;
    return c;
}

template <int BLOCK_N>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
conv_pair_kernel(const __grid_constant__ PairParams p) {
    using C = QCfg<BLOCK_N>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* patches = smem;
    uint8_t* bstages = smem + C::kPatchRegion;
    uint64_t* pfull = (uint64_t*)(bstages + C::kBStages * C::kBHalfBytes);
    uint64_t* pempty = pfull + C::kNumPatch;
    uint64_t* bfull = pempty + C::kNumPatch;
    uint64_t* bempty = bfull + C::kBStages;
    uint64_t* tfull = bempty + C::kBStages;
    uint64_t* tempty = tfull + kAccStages;
    uint32_t* tmem_slot = (uint32_t*)(tempty + kAccStages);
    float* sbias = (float*)((uint8_t*)pfull + C::kBarBytes);

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
    const int lane = threadIdx.x & 31;
    const int rank = (int)cluster_ctarank();            // 0 = leader
    const int cluster_id = blockIdx.x >> 1;
    const int n_clusters = gridDim.x >> 1;
    const int ks = p.ks;
    const int pad = ks >> 1;
    const int patch_rows = kTile + ks - 1;
    const uint32_t patch_bytes = (uint32_t)(kPitch * patch_rows * 128);
    // a 3x3 patch feeds only 3 x 2 x 4 MMAs (~1500 clocks): four buffers in flight to cover the TMA latency; 7x7: three
    const int n_patch = p.n_patch;
    const uint32_t patch_stride = ks == 3 ? C::kPatchBytes3 : C::kPatchBytesMax;

    if (warp == 0 && lane == 0) {
        for (int i = 0; i < p.nprob; ++i) {
            prefetch_tensormap(&p.tmA[i]);
            prefetch_tensormap(&p.tmW[i]);
        }
        for (int s = 0; s < C::kNumPatch; ++s) {
            mbar_init(&pfull[s], 1);
            mbar_init(&pempty[s], kHalves);             // one commit per issuing warp
        }
        for (int s = 0; s < C::kBStages; ++s) {
            mbar_init(&bfull[s], 1);
            mbar_init(&bempty[s], kHalves);
        }
        for (int a = 0; a < kAccStages; ++a) {
            mbar_init(&tfull[a], kHalves);
            mbar_init(&tempty[a], 256);                 // 128 epilogue threads of each CTA (leader's copy is used)
        }
        fence_barrier_init();
    }
    // Both CTAs of the pair must be resident and past their start-up before either issues the paired TMEM
    // allocation: a cta_group::2 alloc issued while the peer CTA is still being launched (its SM busy with blocks of
    // another stream) left the late CTA's own alloc waiting forever (cuda-gdb: peer warp 1 parked in tcgen05.alloc,
    // everybody else at the cluster barrier below).
    cluster_sync_all();
    if (warp == 1) tmem_alloc_2sm(tmem_slot, C::kTmemCols);
    tc_fence_before();
    cluster_sync_all();                                 // barrier inits + TMEM allocation visible in both CTAs
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

    pdl_launch_dependents();                            // the next layer may start its prologue (it waits before touching data)
    if (warp == 6) {
        // ================= patch (A) producer: own tile =================
        int pb = 0;
        uint32_t pphase = 0;
        pdl_wait();                                     // the activations are the previous kernel's output (weights are not)
        if (p.resident) {
            for (int pr = cluster_id; pr < p.total_pairs; pr += n_clusters) {
                const TileCoord tc = decode_pair(p, pr, rank, BLOCK_N);
                mbar_wait(&pempty[pb], pphase ^ 1, 10);
                if (rank == 0) mbar_arrive_expect_tx_elect(&pfull[pb], 2 * C::kResPatchBytes);
                tma_load_4d_2sm_elect(patches + pb * C::kResPatchStride, &p.tmA[tc.pi], &pfull[pb], 0, tc.x0 - pad, tc.y0 - pad,
                                      tc.img);
                pb ^= 1;
                if (pb == 0) pphase ^= 1;
            }
        } else {
            for (int pr = cluster_id; pr < p.total_pairs; pr += n_clusters) {
                const TileCoord tc = decode_pair(p, pr, rank, BLOCK_N);
                const int cin_chunks = p.prob[tc.pi].cin_chunks;
                const CUtensorMap* tmA = &p.tmA[tc.pi];
                for (int cc = 0; cc < cin_chunks; ++cc) {
                    for (int dx = 0; dx < ks; ++dx) {
                        if (chunk_bit(cc * ks + dx) & p.kskip) continue;
                        mbar_wait(&pempty[pb], pphase ^ 1, 10);
                        if (rank == 0) mbar_arrive_expect_tx_elect(&pfull[pb], 2 * patch_bytes);
                        tma_load_4d_2sm_elect(patches + pb * patch_stride, tmA, &pfull[pb], cc * 64, tc.x0 - pad + dx,
                                              tc.y0 - pad, tc.img);
                        if (++pb == n_patch) { pb = 0; pphase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 0) {
        // ================= weight (B) producer: this CTA's half of the N rows =================
        int bs = 0;
        uint32_t bphase = 0;
        if (p.resident) {
            // all taps once, tap t (row-major dy, dx) in stage t; every stage's barrier completes once and is never re-armed
            for (int t = 0; t < ks * ks; ++t) {
                if (rank == 0) mbar_arrive_expect_tx_elect(&bfull[t], 2 * C::kBHalfBytes);
                tma_load_2d_2sm_elect(bstages + t * C::kBHalfBytes, &p.tmW[0], &bfull[t], t * 64, rank * (BLOCK_N / 2));
            }
        } else if (p.bres) {
            // every chunk once, in the order of the MMA walk, packed back to back; one barrier for the lot
            const int cin_chunks = p.prob[0].cin_chunks;
            if (rank == 0) mbar_arrive_expect_tx_elect(&bfull[0], 2 * (uint32_t)p.bres);
            uint32_t off = 0;
            for (int cc = 0; cc < cin_chunks; ++cc)
                for (int i = 0; i < ks * ks; ++i) {
                    const int tap = (i % ks) * ks + (i / ks);
                    const unsigned bit = chunk_bit(cc * ks + i / ks);
                    if (p.kskip & bit) continue;
                    if ((p.khalf_lo | p.khalf_hi) & bit) {
                        tma_load_2d_2sm_elect(bstages + off, &p.tmWh, &bfull[0], (tap * cin_chunks + cc) * 64,
                                              ((p.khalf_hi & bit) ? BLOCK_N / 2 : 0) + rank * (BLOCK_N / 4));
                        off += C::kBHalfBytes / 2;
                    } else {
                        tma_load_2d_2sm_elect(bstages + off, &p.tmW[0], &bfull[0], (tap * cin_chunks + cc) * 64, rank * (BLOCK_N / 2));
                        off += C::kBHalfBytes;
                    }
                }
        } else {
            for (int pr = cluster_id; pr < p.total_pairs; pr += n_clusters) {
                const TileCoord tc = decode_pair(p, pr, rank, BLOCK_N);
                const int cin_chunks = p.prob[tc.pi].cin_chunks;
                const CUtensorMap* tmW = &p.tmW[tc.pi];
                for (int cc = 0; cc < cin_chunks; ++cc) {
                    for (int i = 0; i < ks * ks; ++i) {
                        const int tap = (i % ks) * ks + (i / ks);              // dx outer, dy inner (matches the MMA walk)
                        const unsigned bit = chunk_bit(cc * ks + i / ks);
                        if (p.kskip & bit) continue;
                        mbar_wait(&bempty[bs], bphase ^ 1, 11);
                        if ((p.khalf_lo | p.khalf_hi) & bit) {
                            // half chunk: N/2 weight rows in all, this CTA's quarter at the head of the stage
                            if (rank == 0) mbar_arrive_expect_tx_elect(&bfull[bs], C::kBHalfBytes);
                            tma_load_2d_2sm_elect(bstages + bs * C::kBHalfBytes, &p.tmWh, &bfull[bs], (tap * cin_chunks + cc) * 64,
                                                  tc.n0 + ((p.khalf_hi & bit) ? BLOCK_N / 2 : 0) + rank * (BLOCK_N / 4));
                        } else {
                            if (rank == 0) mbar_arrive_expect_tx_elect(&bfull[bs], 2 * C::kBHalfBytes);
                            tma_load_2d_2sm_elect(bstages + bs * C::kBHalfBytes, tmW, &bfull[bs], (tap * cin_chunks + cc) * 64,
                                                  tc.n0 + rank * (BLOCK_N / 2));
                        }
                        if (++bs == C::kBStages) { bs = 0; bphase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 1 || warp == 7) {
        // ================= MMA issuers (leader CTA only) =================
        // Two warps, one per 128-pixel half of the super-tiles (each half has its own accumulator columns, so the two MMA
        // streams are independent): one thread could not keep up with short-K layers -- ncu on conv1_2 showed the issuing
        // warp never waiting on a barrier while the tensor pipe idled 45 % of the time.  Each warp waits for the same
        // operands and commits its own MMAs, so the empty / accumulator-full barriers count two arrivals.
        const int h = warp == 1 ? 0 : 1;
        if (rank == 0) {
            constexpr uint32_t idesc = make_idesc_2sm(BLOCK_N);
            constexpr uint32_t idesc_half = make_idesc_2sm(BLOCK_N / 2);
            int pb = 0, bs = 0, acc = 0;
            uint32_t pphase = 0, bphase = 0, acc_phase = 0;
            bool first_tile = true;
            for (int pr = cluster_id; pr < p.total_pairs; pr += n_clusters) {
                const TileCoord tc = decode_pair(p, pr, 0, BLOCK_N);
                const QProb& q = p.prob[tc.pi];
                // a half that is outside the image in BOTH tiles of the pair is neither multiplied nor stored
                const int halves = tc.halves | decode_pair(p, pr, 1, BLOCK_N).halves;
                const uint32_t half_off = tc.vsplit ? 8u * kPitch * 128u : 8u * 128u;
                const uint32_t sbo = tc.vsplit ? 1024u : (uint32_t)(kPitch * 128);
                uint32_t accum = 0;
                const bool mine = halves & (1 << h);
                mbar_wait(&tempty[acc], acc_phase ^ 1, 12);               // both epilogues drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * (kHalves * BLOCK_N);
                if (p.resident) {
                    // one 24-column patch: tap (dy, dx) of half h starts (dy * 24 + dx + 8 h) pixels into it (the swizzle
                    // is a function of the absolute shared-memory address, so a start that is not atom aligned needs no
                    // base offset); the weights of tap t wait in stage t
                    mbar_wait(&pfull[pb], pphase, 13);
                    tc_fence_after();
                    const uint32_t patch_addr = smem_u32(patches + pb * C::kResPatchStride);
                    for (int t = 0; t < ks * ks; ++t) {
                        if (first_tile) {
                            mbar_wait(&bfull[t], 0, 14);
                            tc_fence_after();
                        }
                        const int dy = t / ks, dx = t - dy * ks;
                        const uint64_t bdesc = make_desc(smem_u32(bstages + t * C::kBHalfBytes), 1024);
                        if (mine) {
                            const uint64_t adesc = make_desc(patch_addr + (uint32_t)((dy * C::kResPitch + dx + h * 8) * 128),
                                                             C::kResPitch * 128);
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                umma_bf16_2sm_elect(d_tmem + h * BLOCK_N, adesc + 2 * k, bdesc + 2 * k, idesc, accum);
                                accum = 1;
                            }
                        }
                    }
                    first_tile = false;
                    umma_commit_2sm_elect(&pempty[pb]);
                    pb ^= 1;
                    if (pb == 0) pphase ^= 1;
                } else {
                uint32_t boff = 0;                                        // bres: where this chunk's weights sit
                for (int cc = 0; cc < q.cin_chunks; ++cc) {
                    for (int sh = 0; sh < ks; ++sh) {
                        const unsigned bit = chunk_bit(cc * ks + sh);
                        if (p.kskip & bit) continue;
                        const bool half_n = (p.khalf_lo | p.khalf_hi) & bit;
                        const uint32_t idesc_use = half_n ? idesc_half : idesc;
                        const uint32_t dcol = (p.khalf_hi & bit) ? BLOCK_N / 2 : 0;
                        mbar_wait(&pfull[pb], pphase, 13);                // both CTAs' patches have landed
                        tc_fence_after();
                        const uint32_t patch_addr = smem_u32(patches + pb * patch_stride);
                        for (int dy = 0; dy < ks; ++dy) {
                            uint32_t baddr;
                            if (p.bres) {
                                if (first_tile) {
                                    mbar_wait(&bfull[0], 0, 14);          // the whole weight set has landed in both CTAs
                                    tc_fence_after();
                                    first_tile = false;
                                }
                                baddr = smem_u32(bstages) + boff;
                                boff += half_n ? C::kBHalfBytes / 2 : C::kBHalfBytes;
                            } else {
                                mbar_wait(&bfull[bs], bphase, 14);        // both weight halves have landed
                                tc_fence_after();
                                baddr = smem_u32(bstages + bs * C::kBHalfBytes);
                            }
                            const uint64_t bdesc = make_desc(baddr, 1024);
                            if (mine) {
                                const uint64_t adesc = make_desc(patch_addr + (uint32_t)(dy * kPitch * 128) + h * half_off, sbo);
#pragma unroll
                                for (int k = 0; k < 4; ++k) {
                                    // (a half chunk is never the first of a tile: conv_pair_plan checks)
                                    umma_bf16_2sm_elect(d_tmem + h * BLOCK_N + dcol, adesc + 2 * k, bdesc + 2 * k, idesc_use, accum);
                                    accum = 1;
                                }
                            }
                            if (!p.bres) {
                                umma_commit_2sm_elect(&bempty[bs]);
                                if (++bs == C::kBStages) { bs = 0; bphase ^= 1; }
                            }
                        }
                        umma_commit_2sm_elect(&pempty[pb]);
                        if (++pb == n_patch) { pb = 0; pphase ^= 1; }
                    }
                }
                }
                umma_commit_2sm_elect(&tfull[acc]);
                if (++acc == kAccStages) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else if (warp >= 2 && warp <= 5) {
        // ================= epilogue: own 128 TMEM lanes per half =================
        const int quad = warp & 3;
        const int row = quad * 32 + lane;
        const int ep_tid = threadIdx.x - 64;
        int acc = 0;
        uint32_t acc_phase = 0;
        int bias_loaded[kAccStages];
#pragma unroll
        for (int a = 0; a < kAccStages; ++a) bias_loaded[a] = -1;
        for (int pr = cluster_id; pr < p.total_pairs; pr += n_clusters) {
            const TileCoord tc = decode_pair(p, pr, rank, BLOCK_N);
            const QProb& q = p.prob[tc.pi];
            float* bias_s = sbias + acc * BLOCK_N;
            // the bias slice changes only with the problem / n tile: reloading it for every tile put a global load and a
            // barrier at the head of each epilogue, which is what paced the short-K (1x1, 3x3) layers
            const int bias_key = (tc.pi << 16) | tc.n0;
            if (bias_loaded[acc] != bias_key) {
                asm volatile("bar.sync 1, 128;" ::: "memory");       // nobody still reads this slot (two tiles back)
                if (ep_tid < BLOCK_N) bias_s[ep_tid] = __ldg(q.bias + tc.n0 + ep_tid);
                asm volatile("bar.sync 1, 128;" ::: "memory");       // bias visible to the 4 epilogue warps
                bias_loaded[acc] = bias_key;
            }
            const bool relu = q.flags & FLAG_RELU;
            const bool pool = q.flags & FLAG_POOL;
            const bool f32 = q.flags & FLAG_F32;
            const bool poolw = q.flags & FLAG_POOLW;
            const int n_valid = q.cout_store - tc.n0;
            const bool vsplit = tc.vsplit != 0;
            // pixel of accumulator row `row` inside the half: 8 x 16 (side by side) or 16 x 8 (stacked)
            const int tx = vsplit ? (row & 15) : (row & 7);
            const int ty = vsplit ? (row >> 4) : (row >> 3);
            const int pool_dy = vsplit ? 16 : 8;                      // lane distance of the row below

            mbar_wait(&tfull[acc], acc_phase, 15);
            tc_fence_after();
#pragma unroll 1
            for (int h = 0; h < kHalves; ++h) {
                if (!(tc.halves & (1 << h))) break;
                const int x = tc.x0 + (vsplit ? 0 : 8 * h) + tx;
                const int y = tc.y0 + (vsplit ? 8 * h : 0) + ty;
                const bool inside = (x < q.W) && (y < q.H);
                size_t pix;
                bool writer;
                if (poolw) {
                    pix = ((size_t)tc.img * (q.H >> 1) + (y >> 1)) * q.W + x;
                    writer = inside && !(ty & 1);
                } else if (pool) {
                    pix = ((size_t)tc.img * (q.H >> 1) + (y >> 1)) * (q.W >> 1) + (x >> 1);
                    writer = inside && !(tx & 1) && !(ty & 1);
                } else {
                    pix = ((size_t)tc.img * q.H + y) * q.W + x;
                    writer = inside;
                }
                const size_t out_off = pix * q.out_cstride + tc.n0;
                const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + acc * (kHalves * BLOCK_N) + h * BLOCK_N;
                if (poolw) {
                    // wide pixel: columns c and 64 + c are channel c of the even and of the odd image column
#pragma unroll 1
                    for (int c0 = 0; c0 < 64; c0 += 32) {
                        uint32_t v0[32], v1[32];
                        tmem_ld32(taddr + c0, v0);
                        tmem_ld32(taddr + 64 + c0, v1);
                        float f[32];
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const float a = fmaxf(__uint_as_float(v0[j]) + bias_s[c0 + j], 0.f);
                            const float b = fmaxf(__uint_as_float(v1[j]) + bias_s[64 + c0 + j], 0.f);
                            const float m = fmaxf(a, b);
                            f[j] = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, pool_dy));
                        }
                        if (writer) store_bf16x32((__nv_bfloat16*)q.out + out_off + c0, f, 64 - c0);
                    }
                    continue;
                }
#pragma unroll 1
                for (int c0 = 0; c0 < BLOCK_N; c0 += 32) {
                    if (c0 >= n_valid) break;
                    uint32_t v[32];
                    tmem_ld32(taddr + c0, v);
                    float f[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float a = __uint_as_float(v[j]) + bias_s[c0 + j];
                        f[j] = relu ? fmaxf(a, 0.f) : a;
                    }
                    if (pool) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const float m = fmaxf(f[j], __shfl_xor_sync(0xffffffffu, f[j], 1));
                            f[j] = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, pool_dy));
                        }
                    }
                    if (writer) {
                        if (f32) {
                            float* o = (float*)q.out + out_off + c0;
#pragma unroll
                            for (int j = 0; j < 32; j += 4)
                                if (c0 + j < n_valid) *(float4*)(o + j) = make_float4(f[j], f[j + 1], f[j + 2], f[j + 3]);
                        } else {
                            store_bf16x32((__nv_bfloat16*)q.out + out_off + c0, f, n_valid - c0);
                        }
                    }
                }
            }
            tc_fence_before();
            mbar_arrive_cluster(&tempty[acc], 0);                         // release on the leader's barrier
            if (++acc == kAccStages) { acc = 0; acc_phase ^= 1; }
        }
    }

    // the peer's shared memory and TMEM are operands of the leader's MMAs: nobody leaves before both are done
    tc_fence_before();
    cluster_sync_all();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc_2sm(tmem_base, C::kTmemCols);
    }
    // ... and nobody exits before BOTH CTAs have released their TMEM, so that the next cluster scheduled on this TPC
    // never meets a half-released pair allocation.
    cluster_sync_all();
}

// Tile classes and pair counts of one problem (q.H, q.W, q.N set).
void fill_tiling(QProb& q, bool small, bool resident) {
    const int H = q.H, W = q.W, N = q.N;
    q.tile_h = small ? 8 : kTile;
    q.tiles_x = cdiv(W, kTile);
    q.tiles_y = cdiv(H, q.tile_h);
    {
        // 128-pixel halves actually multiplied.  A tile with pixels in both halves costs 256 rows whatever its
        // orientation; the last tile column is split side by side when at most 8 columns remain there, the last tile
        // row stacked when at most 8 rows remain, and their empty half is skipped: columns and rows both round up to 8
        // (41x23: 48x24, 82x46: 88x48, 69x69: 72x72, 23x23: 24x24).  OPB_PAIR_NO_MIXED=1: one orientation per problem
        // (the one with the least padding), i.e. only one of the two edges profits.
        static const char* force = getenv("OPB_PAIR_SPLIT");
        static const char* noskip = getenv("OPB_PAIR_NOSKIP");
        static const bool mixed = getenv("OPB_PAIR_NO_MIXED") == nullptr;
        const long side = (long)cdiv(W, 8) * 8 * cdiv(H, 16) * 16, stacked = (long)cdiv(W, 16) * 16 * cdiv(H, 8) * 8;
        q.vsplit = small ? 1 : (resident ? 0 : (force ? atoi(force) : (stacked < side ? 1 : 0)));   // 24-column patches: side by side only
        q.noskip = noskip ? 1 : 0;
        const bool skip = !small && !q.noskip;
        const bool has_c = skip && (q.tiles_x - 1) * kTile + 8 >= W && (mixed || q.vsplit == 0);
        const bool has_r = skip && (q.tiles_y - 1) * kTile + 8 >= H && !resident && (mixed || q.vsplit == 1);
        q.fx = q.tiles_x - (has_c ? 1 : 0);
        q.fy = q.tiles_y - (has_r ? 1 : 0);
        q.nF = N * q.fx * q.fy;
        q.nC = has_c ? N * q.fy : 0;
        q.nR = has_r ? N * q.tiles_x : 0;
        q.startC = (q.nF + 1) / 2 * 2;
        q.startR = q.startC + (q.nC + 1) / 2 * 2;
        q.m_tiles = q.startR + q.nR;                       // class padding included
        q.m_pairs = (q.m_tiles + 1) / 2;
    }
    // pairs of class F cost two halves, the rest one
    q.n_full_pairs = small ? q.m_pairs : q.startC / 2;
}

// launch order: the full-cost pairs of every problem, then the half-cost pairs of every problem
int order_pairs(PairParams& P) {
    int at = 0;
    for (int i = 0; i < P.nprob; ++i) {
        P.prob[i].pair_begin = at;
        at += P.prob[i].n_full_pairs * P.prob[i].n_tiles_n;
    }
    P.total_full = at;
    for (int i = 0; i < P.nprob; ++i) {
        P.prob[i].edge_begin = at;
        at += (P.prob[i].m_pairs - P.prob[i].n_full_pairs) * P.prob[i].n_tiles_n;
    }
    return at;
}

struct PairLaunch : ConvLaunch {
    PairParams params;
    int grid = 0, block_n = 128;
    void run(cudaStream_t stream) const override;
};

template <int BN>
void launch_pair(const PairLaunch& L, cudaStream_t stream) {
    static bool attr[64] = {};
    if (first_use_on_device(attr)) {
        OPB_CUDA(cudaFuncSetAttribute(conv_pair_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, QCfg<BN>::kSmemBytes));
    }
    // programmatic dependent launch: the kernel's prologue and its weight loads overlap the previous kernel's tail; the
    // patch producer executes griddepcontrol.wait before the first activation load
    launch_pdl(conv_pair_kernel<BN>, L.grid, kThreads, QCfg<BN>::kSmemBytes, stream, L.params);
}

void PairLaunch::run(cudaStream_t stream) const {
    if (block_n == 128) launch_pair<128>(*this, stream);
    else launch_pair<64>(*this, stream);
    OPB_CUDA(cudaGetLastError());
}

}  // namespace

ConvLaunch* conv_pair_plan(const std::vector<ConvOp>& ops, int block_n, int num_sms) {
    OPB_REQUIRE(!ops.empty() && (int)ops.size() <= kConvMaxProblems, "conv_pair: 1..8 problems per launch");
    OPB_REQUIRE(block_n == 64 || block_n == 128, "conv_pair: block_n must be 64 or 128");
    auto L = std::make_unique<PairLaunch>();
    PairParams& P = L->params;
    memset(&P, 0, sizeof(P));
    P.nprob = (int)ops.size();
    P.ks = ops[0].ks;
    P.kskip = ops[0].kskip;
    {
        static const char* np = getenv("OPB_PAIR_PATCHES");
        P.n_patch = P.ks == 3 ? 4 : 3;
        if (np && atoi(np) >= 2 && atoi(np) <= P.n_patch) P.n_patch = atoi(np);
    }
    P.khalf_lo = ops[0].khalf_lo;
    P.khalf_hi = ops[0].khalf_hi;
    if (P.khalf_lo | P.khalf_hi) {
        OPB_REQUIRE(block_n == 128 && !(P.khalf_lo & P.khalf_hi) && !((P.khalf_lo | P.khalf_hi) & P.kskip),
                    "conv_pair: half chunks need the 128-wide N tile and disjoint masks");
        int first = 0;
        while ((P.kskip >> first) & 1) ++first;
        OPB_REQUIRE(!(((P.khalf_lo | P.khalf_hi) >> first) & 1), "conv_pair: the first chunk of a tile must span the whole N tile");
        const ConvOp& op = ops[0];
        const cuuint64_t K = (cuuint64_t)op.ks * op.ks * op.in.c;
        cuuint64_t wdims[2] = {K, (cuuint64_t)op.cout_pad};
        cuuint64_t wstr[1] = {K * 2};
        cuuint32_t wbox[2] = {64, (cuuint32_t)(block_n / 4)};
        tensor_map_encode_bf16(&P.tmWh, (void*)op.w, 2, wdims, wstr, wbox);
    }
    OPB_REQUIRE(P.ks == 3 || P.ks == 7, "conv_pair: kernel size 3 or 7");
    // Small launches (a 640x480 frame at scale 0.5 gives 4 super-tiles per stage layer): when full 16x16 super-tiles
    // would occupy at most a quarter of the CTA pairs the GPU holds, every CTA takes one 16x8 half instead -- twice the
    // pairs, half the UMMAs per CTA, i.e. half the latency of the layer.  Pooling layers keep 16x16 (2x2 windows).
    bool small = getenv("OPB_NO_HALF_TILES") == nullptr;
    {
        long full_pairs = 0;
        for (const ConvOp& op : ops) {
            full_pairs += (long)((cdiv(op.in.w, kTile) * cdiv(op.in.h, kTile) * op.in.n + 1) / 2) * (op.cout_pad / block_n);
            if (op.pool || op.pool_wide) small = false;
        }
        if (full_pairs * 4 > num_sms / 2) small = false;
    }
    // resident mode (opt-in, OPB_CONV12_RESIDENT=1): a 3x3 layer on 64 input channels with one weight set and one 64-wide
    // N tile (conv1_2 at every scale).  Measured on B200 at batch 8: 1.63 ms against 1.50 ms for the default path
    // (654 vs 711 TFLOP/s): the layer is bound by shared-memory operand reads, not by L2 -> SM traffic, and the
    // unaligned swizzle atoms of the single 24-column patch cost more wavefronts than the 2.7x smaller traffic saves.
    bool resident = block_n == 64 && P.ks == 3 && !small && getenv("OPB_CONV12_RESIDENT") != nullptr;
    for (const ConvOp& op : ops)
        resident = resident && op.in.c == 64 && op.cout_pad == 64 && op.w == ops[0].w;
    P.resident = resident ? 1 : 0;
    int pairs = 0;
    for (int i = 0; i < P.nprob; ++i) {
        const ConvOp& op = ops[i];
        OPB_REQUIRE(op.ks == P.ks, "conv_pair: grouped problems must share the kernel size");
        OPB_REQUIRE(op.in.elem == 2 && op.in.c % 64 == 0, "conv_pair: input must be bf16 with C % 64 == 0");
        OPB_REQUIRE(op.in.cstride % 8 == 0 && op.in.coff % 8 == 0, "conv_pair: input slice must be 16-byte aligned");
        OPB_REQUIRE(op.cout_pad % block_n == 0 && op.cout_store % 8 == 0 && op.cout_store <= op.cout_pad,
                    "conv_pair: bad output channel padding");
        OPB_REQUIRE(op.out.elem == 2 || op.out.elem == 4, "conv_pair: output must be bf16 or fp32");
        OPB_REQUIRE((op.out.coff * op.out.elem) % 16 == 0 && (op.out.cstride * op.out.elem) % 16 == 0,
                    "conv_pair: output slice must be 16-byte aligned");
        const int H = op.in.h, W = op.in.w, N = op.in.n;
        OPB_REQUIRE(op.kskip == ops[0].kskip && op.khalf_lo == ops[0].khalf_lo && op.khalf_hi == ops[0].khalf_hi &&
                        ((op.khalf_lo | op.khalf_hi) == 0 || op.w == ops[0].w),
                    "conv_pair: grouped problems must share the zero-chunk masks (and the weights when there are half chunks)");
        if (op.pool_wide) {
            OPB_REQUIRE(block_n == 128 && op.cout_pad == 128 && op.in.c == 128 && P.ks == 3 && op.relu && !op.pool && H % 2 == 0 &&
                            op.out.elem == 2,
                        "conv_pair: wide-pixel pooled form is 128 -> 128 columns, 3x3, ReLU, even rows, bf16 out");
            OPB_REQUIRE(op.out.h == H / 2 && op.out.w == W && op.out.n == N && op.out.c == 64, "conv_pair: wide-pixel output dims");
        } else if (op.pool) {
            OPB_REQUIRE(H % 2 == 0 && W % 2 == 0 && op.relu, "conv_pair: fused pool needs even dims and ReLU");
            OPB_REQUIRE(op.out.h == H / 2 && op.out.w == W / 2 && op.out.n == N, "conv_pair: pooled output dims");
        } else {
            OPB_REQUIRE(op.out.h == H && op.out.w == W && op.out.n == N, "conv_pair: output dims");
        }
        QProb& q = P.prob[i];
        q.out = op.out.ptr();
        q.bias = op.bias;
        q.H = H; q.W = W; q.N = N;
        q.out_cstride = op.out.cstride;
        q.cout_store = op.cout_store;
        q.n_tiles_n = op.cout_pad / block_n;
        q.cin_chunks = op.in.c / 64;
        q.flags = (op.relu ? FLAG_RELU : 0) | (op.out.elem == 4 ? FLAG_F32 : 0) | (op.pool ? FLAG_POOL : 0) |
                  (op.pool_wide ? FLAG_POOLW : 0);
        fill_tiling(q, small, resident);
        pairs += q.m_pairs * q.n_tiles_n;

        cuuint64_t adims[4] = {(cuuint64_t)op.in.c, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
        cuuint64_t astr[3] = {(cuuint64_t)op.in.cstride * 2, (cuuint64_t)op.in.cstride * 2 * W,
                              (cuuint64_t)op.in.cstride * 2 * W * H};
        cuuint32_t abox[4] = {64, (cuuint32_t)(resident ? QCfg<64>::kResPitch : kPitch), (cuuint32_t)(kTile + P.ks - 1), 1};
        tensor_map_encode_bf16(&P.tmA[i], op.in.ptr(), 4, adims, astr, abox);
        const cuuint64_t K = (cuuint64_t)op.ks * op.ks * op.in.c;
        cuuint64_t wdims[2] = {K, (cuuint64_t)op.cout_pad};
        cuuint64_t wstr[1] = {K * 2};
        cuuint32_t wbox[2] = {64, (cuuint32_t)(block_n / 2)};
        tensor_map_encode_bf16(&P.tmW[i], (void*)op.w, 2, wdims, wstr, wbox);
    }
    // weights resident for the whole kernel: one weight set, one N tile, and every chunk fits the weight stages
    if (!resident && getenv("OPB_NO_BRES") == nullptr) {
        bool same = true;
        for (const ConvOp& op : ops) same = same && op.w == ops[0].w && op.cout_pad == block_n && op.in.c == ops[0].in.c;
        long bytes = 0;
        for (int cc = 0; cc < ops[0].in.c / 64; ++cc)
            for (int dx = 0; dx < P.ks; ++dx) {
                const unsigned bit = chunk_bit(cc * P.ks + dx);
                if (P.kskip & bit) continue;
                bytes += (long)P.ks * (((P.khalf_lo | P.khalf_hi) & bit) ? (block_n / 4) * 128 : (block_n / 2) * 128);
            }
        if (same && bytes <= (long)9 * (block_n / 2) * 128) P.bres = (int)bytes;
    }
    OPB_REQUIRE(order_pairs(P) == pairs, "conv_pair: pair order");
    P.total_pairs = pairs;
    L->tiles = pairs * 2;
    L->half_tiles = small;
    L->weights_resident = P.bres > 0;
    L->block_n = block_n;
    const int clusters = pairs < num_sms / 2 ? pairs : num_sms / 2;
    L->grid = clusters * 2;
    return L.release();
}

// Host only: the tile list of one problem as the kernel decodes it -- 8 ints per (pair, rank): image, x0, y0, n0, real,
// halves, vsplit, full-cost flag.  For the CPU test of the tiling (exact cover, pairs share an orientation).
int conv_pair_debug_tiles(int n, int h, int w, int n_tiles_n, int small, int* out, int cap) {
    PairParams P;
    memset(&P, 0, sizeof(P));
    P.nprob = 1;
    P.ks = 3;
    QProb& q = P.prob[0];
    q.H = h; q.W = w; q.N = n;
    q.n_tiles_n = n_tiles_n;
    fill_tiling(q, small != 0, false);
    P.total_pairs = order_pairs(P);
    int written = 0;
    for (int pr = 0; pr < P.total_pairs; ++pr)
        for (int rank = 0; rank < 2; ++rank) {
            const TileCoord c = decode_pair(P, pr, rank, 128);
            if ((written + 1) * 8 > cap) return -1;
            int* o = out + written * 8;
            o[0] = c.img; o[1] = c.x0; o[2] = c.y0; o[3] = c.n0; o[4] = c.real ? 1 : 0; o[5] = c.halves; o[6] = c.vsplit;
            o[7] = pr < P.total_full ? 1 : 0;
            ++written;
        }
    return written;
}

}  // namespace opb
