// Network definitions (src/model.py:25-214), checkpoint repacking (src/util.py:36-40, src/body.py:20-21) and
// the per-shape execution plan that strings the convolution kernels together.
//
// Device activation layout: NHWC bf16.  The stage inputs `torch.cat([L1, L2, feat], 1)` (src/model.py:112,
// 116,...; hand: :200) are never materialised by a copy: one 192-channel concat buffer per scale holds
//     [ feat 0..127 | PAF 128..165 (+2 zero) | heat 168..186 (+5 zero) ]        (body, 185 real channels)
//     [ feat 0..127 | heat 128..149 (+2 zero) | 40 zero channels ]               (hand, 150 real channels)
// conv4_4_CPM / conv5_3_CPM write the feature slice once, every stage's last 1x1 conv writes its slice in its
// epilogue, and the Mconv1 weights are permuted on the host to this channel order.
#include "net.cuh"
#include <cmath>
#include <cstring>
#include <cstdlib>

namespace opb {

// ------------------------------------------------------------------------------------------------
// architecture tables
// ------------------------------------------------------------------------------------------------
static std::vector<LayerSpec> make_specs(int kind) {
    std::vector<LayerSpec> v;
    auto add = [&](const std::string& n, int ci, int co, int k, bool relu = true, bool pool = false) {
        v.push_back({n, ci, co, k, relu, pool});
    };
    add("conv1_1", 3, 64, 3);
    add("conv1_2", 64, 64, 3, true, true);
    add("conv2_1", 64, 128, 3);
    add("conv2_2", 128, 128, 3, true, true);
    add("conv3_1", 128, 256, 3);
    add("conv3_2", 256, 256, 3);
    add("conv3_3", 256, 256, 3);
    add("conv3_4", 256, 256, 3, true, true);
    add("conv4_1", 256, 512, 3);
    add("conv4_2", 512, 512, 3);
    char buf[64];
    if (kind == OPB_NET_BODY) {
        add("conv4_3_CPM", 512, 256, 3);
        add("conv4_4_CPM", 256, 128, 3);
        for (int b = 1; b <= 2; ++b) {
            const int co = b == 1 ? 38 : 19;
            for (int i = 1; i <= 3; ++i) {
                snprintf(buf, sizeof buf, "conv5_%d_CPM_L%d", i, b);
                add(buf, 128, 128, 3);
            }
            snprintf(buf, sizeof buf, "conv5_4_CPM_L%d", b);
            add(buf, 128, 512, 1);
            snprintf(buf, sizeof buf, "conv5_5_CPM_L%d", b);
            add(buf, 512, co, 1, false);
        }
        for (int s = 2; s <= 6; ++s)
            for (int b = 1; b <= 2; ++b) {
                const int co = b == 1 ? 38 : 19;
                for (int i = 1; i <= 5; ++i) {
                    snprintf(buf, sizeof buf, "Mconv%d_stage%d_L%d", i, s, b);
                    add(buf, i == 1 ? 185 : 128, 128, 7);
                }
                snprintf(buf, sizeof buf, "Mconv6_stage%d_L%d", s, b);
                add(buf, 128, 128, 1);
                snprintf(buf, sizeof buf, "Mconv7_stage%d_L%d", s, b);
                // src/model.py:30-33 omits 'Mconv7_stage6_L2' from no_relu_layers: the final heat map IS ReLU'd
                add(buf, 128, co, 1, s == 6 && b == 2);
            }
    } else {
        add("conv4_3", 512, 512, 3);
        add("conv4_4", 512, 512, 3);
        add("conv5_1", 512, 512, 3);
        add("conv5_2", 512, 512, 3);
        add("conv5_3_CPM", 512, 128, 3);
        add("conv6_1_CPM", 128, 512, 1);
        add("conv6_2_CPM", 512, 22, 1, false);
        for (int s = 2; s <= 6; ++s) {
            for (int i = 1; i <= 5; ++i) {
                snprintf(buf, sizeof buf, "Mconv%d_stage%d", i, s);
                add(buf, i == 1 ? 150 : 128, 128, 7);
            }
            snprintf(buf, sizeof buf, "Mconv6_stage%d", s);
            add(buf, 128, 128, 1);
            snprintf(buf, sizeof buf, "Mconv7_stage%d", s);
            add(buf, 128, 22, 1, false);
        }
    }
    return v;
}

const std::vector<LayerSpec>& layer_specs(int kind) {
    static const std::vector<LayerSpec> body = make_specs(OPB_NET_BODY);
    static const std::vector<LayerSpec> hand = make_specs(OPB_NET_HAND);
    return kind == OPB_NET_BODY ? body : hand;
}

// ------------------------------------------------------------------------------------------------
// device pool
// ------------------------------------------------------------------------------------------------
void* DevPool::alloc(size_t n, bool zero) {
    void* p = nullptr;
    if (n == 0) n = 16;
    OPB_CUDA(cudaMalloc(&p, n));
    ptrs.push_back(p);
    bytes += n;
    if (zero) {
        // The fill runs on the legacy default stream, which the library's non-blocking streams do not order against:
        // wait for it here (this stream only -- no device-wide synchronisation), so that no kernel launched afterwards
        // on any stream can be overtaken by it.
        OPB_CUDA(cudaMemsetAsync(p, 0, n, cudaStreamLegacy));
        OPB_CUDA(cudaStreamSynchronize(cudaStreamLegacy));
    }
    return p;
}
void DevPool::release() {
    for (void* p : ptrs) cudaFree(p);
    ptrs.clear();
}

NetPlan::~NetPlan() {
    for (auto* l : launches) conv_tc_plan_free(l);
}

// ------------------------------------------------------------------------------------------------
// checkpoint repack
// ------------------------------------------------------------------------------------------------
static inline int round_up(int a, int b) { return (a + b - 1) / b * b; }

// device input channel -> reference input channel (or -1 for a zero pad channel)
static std::vector<int> input_channel_map(int kind, const LayerSpec& s) {
    std::vector<int> m;
    if (s.cin == 185 && kind == OPB_NET_BODY) {          // cat([PAF 38, heat 19, feat 128])  src/model.py:112
        m.assign(192, -1);
        for (int c = 0; c < 128; ++c) m[c] = 57 + c;
        for (int c = 0; c < 38; ++c) m[128 + c] = c;
        for (int c = 0; c < 19; ++c) m[168 + c] = 38 + c;
    } else if (s.cin == 150 && kind == OPB_NET_HAND) {   // cat([heat 22, feat 128])  src/model.py:200
        m.assign(192, -1);
        for (int c = 0; c < 128; ++c) m[c] = 22 + c;
        for (int c = 0; c < 22; ++c) m[128 + c] = c;
    } else {
        m.resize(s.cin);
        for (int c = 0; c < s.cin; ++c) m[c] = c;
    }
    return m;
}

static float bf16_round(float f) { return __bfloat162float(__float2bfloat16_rn(f)); }

// A 3x3 layer on 64 channels gives a 64-wide N tile, and a tcgen05 MMA of N = 64 spends as long fetching its A operand
// from shared memory as one of N = 128 while doing half the arithmetic (conv1_2 ran at 0.48 of the rate of the N = 128
// layers).  Pairing horizontally adjacent pixels turns the layer into a 128 -> 128 channel one on an image of half the
// width: input "channel" (parity pi, c) of wide pixel i is channel c of column 2 i + pi, output column (po, co) is channel
// co of column 2 i + po, and the weight of wide tap (dy, di) is the original tap dx = 2 di + pi - po where that is in
// [-1, 1] and zero elsewhere.  Of the 6 (di, pi) chunks of 64 input channels per dy, (di = -1, pi = 0) and (di = +1, pi = 1)
// are entirely zero and are skipped (kskip); (di = -1, pi = 1) feeds the even output column only and (di = +1, pi = 0) the
// odd one only, and run as MMAs of N = 64 into that half of the accumulator (khalf_lo / khalf_hi).  Per dy that leaves
// two MMAs of N = 128 and two of N = 64 for three taps of useful work (6 N=64-equivalents issued for 6 useful).
// The arithmetic per output element is unchanged: the same nine 64-term dot products accumulate in fp32 in the same
// chunk order (dx outer, dy inner), zero weights add exact zeros.
void wide_pool_weights(const float* weight, const float* bias, std::vector<__nv_bfloat16>& w_wide, std::vector<float>& b_wide) {
    const size_t K = 9 * 128;
    w_wide.assign(128 * K, __float2bfloat16_rn(0.f));
    b_wide.assign(128, 0.f);
    for (int po = 0; po < 2; ++po)
        for (int co = 0; co < 64; ++co) {
            b_wide[po * 64 + co] = bias[co];
            for (int dy = 0; dy < 3; ++dy)
                for (int di = 0; di < 3; ++di)
                    for (int pi = 0; pi < 2; ++pi) {
                        const int dx = 2 * (di - 1) + pi - po;           // signed original column tap
                        if (dx < -1 || dx > 1) continue;
                        const int t = dy * 3 + dx + 1;
                        for (int c = 0; c < 64; ++c)
                            w_wide[(size_t)(po * 64 + co) * K + (size_t)(dy * 3 + di) * 128 + pi * 64 + c] =
                                __float2bfloat16_rn(weight[((size_t)co * 64 + c) * 9 + t]);
                    }
        }
}
bool wide_pool_ok(const ConvOp& b) {
    return b.ks == 3 && b.pool && b.relu && b.in.c == 64 && b.in.cstride == 64 && b.in.coff == 0 && b.in.elem == 2 &&
           b.in.w % 2 == 0 && b.in.h % 2 == 0 && b.out.elem == 2 && b.out.c == 64 && b.out.cstride == 64 && b.out.coff == 0;
}
ConvOp wide_pool_op(const ConvOp& base, const __nv_bfloat16* w_wide, const float* b_wide) {
    OPB_REQUIRE(wide_pool_ok(base), "wide_pool_op: 64 -> 64 channel 3x3 + pool on contiguous bf16 tensors of even size");
    ConvOp op = base;
    op.in.w = base.in.w / 2;
    op.in.c = op.in.cstride = 128;
    op.w = w_wide;
    op.bias = b_wide;
    op.cout_pad = op.cout_store = 128;
    op.pool = false;
    op.pool_wide = true;
    op.kskip = (1u << (0 * 3 + 0)) | (1u << (1 * 3 + 2));     // (pi 0, di -1) and (pi 1, di +1)
    if (getenv("OPB_WIDE_FULL_N") == nullptr) {
        op.khalf_lo = 1u << (1 * 3 + 0);                      // (pi 1, di -1) feeds the even output column only
        op.khalf_hi = 1u << (0 * 3 + 2);                      // (pi 0, di +1) the odd one only
    }
    return op;
}

void finalize_net(opb_net* net) {
    const auto& specs = layer_specs(net->kind);
    for (const auto& s : specs) {
        auto it = net->host.find(s.name);
        if (it == net->host.end())
            throw Error(OPB_ERR_MISSING_LAYER, "checkpoint has no layer '" + s.name + "' (KeyError in util.transfer)");
        const HostLayer& h = it->second;
        if (h.cout != s.cout || h.cin != s.cin || h.k != s.k)
            throw Error(OPB_ERR_INVALID, "layer '" + s.name + "' has the wrong shape");
    }
    OPB_CUDA(cudaSetDevice(net->ctx->device));
    auto dalloc = [&](size_t bytes) {
        void* p = nullptr;
        OPB_CUDA(cudaMalloc(&p, bytes));
        net->owned.push_back(p);
        return p;
    };
    for (const auto& s : specs) {
        const HostLayer& h = net->host[s.name];
        DevLayer d;
        d.k = s.k;
        d.relu = s.relu;
        if (s.cin == 3) {
            // conv1_1: [tap*3 + c][cout] fp32, values rounded to bf16 (the compute precision of the path)
            std::vector<float> w(27 * 64);
            for (int co = 0; co < 64; ++co)
                for (int c = 0; c < 3; ++c)
                    for (int t = 0; t < 9; ++t) w[(t * 3 + c) * 64 + co] = bf16_round(h.w[((size_t)co * 3 + c) * 9 + t]);
            d.w_first = (float*)dalloc(w.size() * 4);
            OPB_CUDA(cudaMemcpy(d.w_first, w.data(), w.size() * 4, cudaMemcpyHostToDevice));
            d.cout_pad = d.cout_store = 64;
            d.cin_dev = 3;
            d.bias = (float*)dalloc(64 * 4);
            OPB_CUDA(cudaMemcpy(d.bias, h.b.data(), 64 * 4, cudaMemcpyHostToDevice));
        } else {
            const std::vector<int> cmap = input_channel_map(net->kind, s);
            d.cin_dev = (int)cmap.size();
            OPB_REQUIRE(d.cin_dev % 64 == 0, "device input channels must be a multiple of 64");
            d.block_n = (s.cout == 64 || s.cout < 64) ? 64 : 128;
            d.cout_pad = round_up(s.cout, d.block_n);
            d.cout_store = round_up(s.cout, 8);
            const int taps = s.k * s.k;
            const size_t K = (size_t)taps * d.cin_dev;
            std::vector<__nv_bfloat16> w((size_t)d.cout_pad * K, __float2bfloat16_rn(0.f));
            for (int co = 0; co < s.cout; ++co)
                for (int t = 0; t < taps; ++t)
                    for (int c = 0; c < d.cin_dev; ++c) {
                        const int rc = cmap[c];
                        if (rc < 0) continue;
                        w[(size_t)co * K + (size_t)t * d.cin_dev + c] =
                            __float2bfloat16_rn(h.w[((size_t)co * s.cin + rc) * taps + t]);
                    }
            d.w = (__nv_bfloat16*)dalloc(w.size() * 2);
            OPB_CUDA(cudaMemcpy(d.w, w.data(), w.size() * 2, cudaMemcpyHostToDevice));
            std::vector<float> b(d.cout_pad, 0.f);
            for (int co = 0; co < s.cout; ++co) b[co] = h.b[co];
            d.bias = (float*)dalloc(b.size() * 4);
            OPB_CUDA(cudaMemcpy(d.bias, b.data(), b.size() * 4, cudaMemcpyHostToDevice));
            if (s.k == 3 && s.cin == 64 && s.cout == 64 && s.pool_after) {
                std::vector<__nv_bfloat16> ww;
                std::vector<float> bw;
                wide_pool_weights(h.w.data(), h.b.data(), ww, bw);
                d.w_wide = (__nv_bfloat16*)dalloc(ww.size() * 2);
                OPB_CUDA(cudaMemcpy(d.w_wide, ww.data(), ww.size() * 2, cudaMemcpyHostToDevice));
                d.bias_wide = (float*)dalloc(bw.size() * 4);
                OPB_CUDA(cudaMemcpy(d.bias_wide, bw.data(), bw.size() * 4, cudaMemcpyHostToDevice));
            }
        }
        net->dev[s.name] = d;
    }
    net->host.clear();
    net->finalized = true;
}

// ------------------------------------------------------------------------------------------------
// execution plan
// ------------------------------------------------------------------------------------------------
namespace {

struct Builder {
    opb_net* net;
    NetPlan* plan;
    bool fuse_pool;
    int conv_impl;          // -1: per-tap tiles everywhere, 0 / 1: patch-resident MODE 0 / 1, 2: CTA-pair kernel (ks > 1)
    TensorView act(int n, int h, int w, int c, int elem = 2, bool zero = false) {
        TensorView t;
        t.n = n; t.h = h; t.w = w; t.c = c; t.cstride = c; t.coff = 0; t.elem = elem;
        t.base = plan->pool.alloc((size_t)n * h * w * c * elem, zero);
        return t;
    }
    static TensorView slice(const TensorView& t, int coff, int c) {
        TensorView s = t;
        s.coff = t.coff + coff;
        s.c = c;
        return s;
    }
    // one grouped tensor-core launch; ins/outs parallel vectors, all with the same layer kernel size/block_n
    void conv_group(const std::vector<std::string>& names, const std::vector<int>& scales, const std::vector<TensorView>& ins,
                    const std::vector<TensorView>& outs, bool pool) {
        size_t i = 0;
        while (i < names.size()) {
            std::vector<ConvOp> ops;
            const int bn = net->dev.at(names[i]).block_n;
            const size_t first = i;
            double gf = 0;
            for (; i < names.size() && (int)ops.size() < kConvMaxProblems; ++i) {
                const DevLayer& d = net->dev.at(names[i]);
                if (d.block_n != bn) break;
                gf += add_flops(names[i], ins[i]);
                ConvOp op;
                op.in = ins[i];
                op.out = outs[i];
                op.w = d.w;
                op.bias = d.bias;
                op.cout_pad = d.cout_pad;
                op.cout_store = d.cout_store;
                op.ks = d.k;
                op.relu = d.relu;
                op.pool = pool;
                OPB_REQUIRE(op.in.c == d.cin_dev, "plan: input channel mismatch for " + names[i]);
                ops.push_back(op);
            }
            StepInfo info;
            info.kind = kStepConv;
            info.pool = pool;
            for (size_t j = 0; j < ops.size(); ++j)
                info.probs.push_back({names[first + j], "", scales[first + j], ops[j].in, ops[j].out});
            // 3x3 / 7x7 layers run patch-resident (conv_patch.cu); 1x1 layers (and OPB_CONV_IMPL=tap) per-tap tiles
            // Small problems (one 640x480 frame at scale 0.5 gives 4 super-tiles per stage layer) leave most SMs idle and
            // their latency is the depth of one tile's K loop: halve the N tile so that twice as many CTA pairs share
            // the work and every UMMA is half as long.
            int bn_run = bn;
            // conv1_2: wide-pixel form (wide_pool_weights above); OPB_NO_WIDE_CONV12=1 keeps the N = 64 launch
            if (conv_impl == 2 && pool && getenv("OPB_NO_WIDE_CONV12") == nullptr) {
                bool wide = true;
                for (size_t j = 0; j < ops.size(); ++j)
                    wide = wide && net->dev.at(names[first + j]).w_wide != nullptr && wide_pool_ok(ops[j]);
                if (wide) {
                    for (size_t j = 0; j < ops.size(); ++j) {
                        const DevLayer& d = net->dev.at(names[first + j]);
                        ops[j] = wide_pool_op(ops[j], d.w_wide, d.bias_wide);
                    }
                    bn_run = 128;
                    info.wide = true;
                }
            }
            if (ops[0].ks > 1 && conv_impl == 2 && bn == 128 && getenv("OPB_NO_SMALL_BN") == nullptr) {
                long clusters = 0;
                for (const ConvOp& op : ops)
                    clusters += (long)((cdiv(op.in.w, 16) * cdiv(op.in.h, 16) * op.in.n + 1) / 2) * (op.cout_pad / 128);
                if (clusters * 4 <= net->ctx->num_sms) bn_run = 64;
            }
            ConvLaunch* L = (ops[0].ks > 1 && conv_impl == 2) ? conv_pair_plan(ops, bn_run, net->ctx->num_sms)
                            : (ops[0].ks > 1 && conv_impl >= 0) ? conv_patch_plan(ops, bn, net->ctx->num_sms, conv_impl)
                                                                : conv_tc_plan(ops, bn, net->ctx->num_sms);
            plan->launches.push_back(L);
            plan->steps.push_back([L](cudaStream_t s) { conv_tc_plan_run(L, s); });
            plan->step_names.push_back(std::string(bn_run == 128 ? "conv_tc128:" : "conv_tc64:") + names[first]);   // the N tile that runs
            info.block_n = bn_run;
            info.pair = ops[0].ks > 1 && conv_impl == 2;
            info.half_tiles = L->half_tiles;
            info.weights_resident = L->weights_resident;
            plan->step_info.push_back(info);
            plan->step_gflop.push_back(gf);
            plan->kernel_launches += 1;
        }
    }
    // Mconv6 + Mconv7 of a refinement stage as one fused launch (conv_tail.cu); OPB_NO_FUSE_TAILS=1: two grouped launches.
    bool tail_group(const std::vector<std::string>& n6, const std::vector<std::string>& n7, const std::vector<int>& scales,
                    const std::vector<TensorView>& ins, const std::vector<TensorView>& outs) {
        static const bool fuse = getenv("OPB_NO_FUSE_TAILS") == nullptr;
        if (!fuse) return false;
        std::vector<TailOp> ops;
        double gf = 0;
        for (size_t i = 0; i < n6.size(); ++i) {
            const DevLayer& a = net->dev.at(n6[i]);
            const DevLayer& b = net->dev.at(n7[i]);
            if (a.k != 1 || b.k != 1 || a.cin_dev != 128 || a.cout_pad != 128 || a.cout_store != 128 || !a.relu ||
                b.cin_dev != 128 || b.cout_pad != 64)
                return false;
            TailOp op;
            op.in = ins[i];
            op.out = outs[i];
            op.w1 = a.w; op.b1 = a.bias;
            op.w2 = b.w; op.b2 = b.bias;
            op.cout_pad2 = b.cout_pad;
            op.cout_store = b.cout_store;
            op.relu2 = b.relu;
            ops.push_back(op);
        }
        if (!conv_tail_supported(ops)) return false;
        for (size_t i = 0; i < n6.size(); ++i) {
            gf += add_flops(n6[i], ins[i]);
            gf += add_flops(n7[i], ins[i]);
        }
        ConvLaunch* L = conv_tail_plan(ops, net->ctx->num_sms);
        plan->launches.push_back(L);
        plan->steps.push_back([L](cudaStream_t s) { conv_tc_plan_run(L, s); });
        plan->step_names.push_back("conv_tail:" + n6[0]);
        plan->step_gflop.push_back(gf);
        plan->kernel_launches += 1;
        tail_info(kStepTail, n6, n7, scales, ins, outs);
        return true;
    }
    // conv5_4 + conv5_5 of stage 1 (hand: conv6_1 + conv6_2) as one fused launch with the 512-channel intermediate kept on
    // the SM (conv_tail.cu, wide variant); OPB_NO_FUSE_WIDE=1: two grouped launches through HBM.
    bool wide_tail_group(const std::vector<std::string>& n4, const std::vector<std::string>& n5, const std::vector<int>& scales,
                         const std::vector<TensorView>& ins, const std::vector<TensorView>& outs) {
        static const bool fuse = getenv("OPB_NO_FUSE_WIDE") == nullptr && getenv("OPB_NO_FUSE_TAILS") == nullptr;
        if (!fuse) return false;
        std::vector<TailOp> ops;
        double gf = 0;
        for (size_t i = 0; i < n4.size(); ++i) {
            const DevLayer& a = net->dev.at(n4[i]);
            const DevLayer& b = net->dev.at(n5[i]);
            if (a.k != 1 || b.k != 1 || a.cin_dev != 128 || a.cout_pad != 512 || a.cout_store != 512 || !a.relu ||
                b.cin_dev != 512 || b.cout_pad != 64)
                return false;
            TailOp op;
            op.in = ins[i];
            op.out = outs[i];
            op.w1 = a.w; op.b1 = a.bias;
            op.w2 = b.w; op.b2 = b.bias;
            op.cout_pad2 = b.cout_pad;
            op.cout_store = b.cout_store;
            op.relu2 = b.relu;
            ops.push_back(op);
        }
        if (!conv_tail_wide_supported(ops)) return false;
        for (size_t i = 0; i < n4.size(); ++i) {
            gf += add_flops(n4[i], ins[i]);
            gf += add_flops(n5[i], ins[i]);
        }
        ConvLaunch* L = conv_tail_wide_plan(ops, net->ctx->num_sms);
        plan->launches.push_back(L);
        plan->steps.push_back([L](cudaStream_t s) { conv_tc_plan_run(L, s); });
        plan->step_names.push_back("conv_tail:" + n4[0]);
        plan->step_gflop.push_back(gf);
        plan->kernel_launches += 1;
        tail_info(kStepTailWide, n4, n5, scales, ins, outs);
        return true;
    }
    void tail_info(int kind, const std::vector<std::string>& n1, const std::vector<std::string>& n2, const std::vector<int>& scales,
                   const std::vector<TensorView>& ins, const std::vector<TensorView>& outs) {
        StepInfo info;
        info.kind = kind;
        info.block_n = 128;
        for (size_t i = 0; i < n1.size(); ++i) info.probs.push_back({n1[i], n2[i], scales[i], ins[i], outs[i]});
        plan->step_info.push_back(info);
    }
    // algorithmic FLOPs of one layer on one input (un-padded channel counts, SURVEY.md 8d)
    double add_flops(const std::string& name, const TensorView& in) {
        for (const auto& s : layer_specs(net->kind))
            if (s.name == name) {
                const double gf = 2.0 * s.cout * s.cin * s.k * s.k * (double)in.pixels() * 1e-9;
                plan->gflop += gf;
                return gf;
            }
        return 0.0;
    }
};

}  // namespace

int default_conv_impl() {
    const char* e = getenv("OPB_CONV_IMPL");
    if (e && !strcmp(e, "tap")) return -1;
    if (e && !strcmp(e, "patch0")) return 0;
    if (e && !strcmp(e, "patch1")) return 1;
    if (e && !strcmp(e, "pair")) return 2;
    return kDefaultConvImpl;
}

std::unique_ptr<NetPlan> build_net_plan(opb_net* net, const std::vector<NetShape>& shapes) {
    OPB_REQUIRE(net->finalized, "net not finalized");
    OPB_REQUIRE(!shapes.empty() && (int)shapes.size() <= kMaxScales, "1..8 scales per plan");
    auto plan = std::make_unique<NetPlan>();
    plan->shapes = shapes;
    Builder B{net, plan.get(), getenv("OPB_NO_FUSE_POOL") == nullptr, default_conv_impl()};
    const int S = (int)shapes.size();
    const bool body = net->kind == OPB_NET_BODY;
    std::vector<TensorView> cur(S);

    // ---- conv1_1 (CUDA cores) ----
    for (int s = 0; s < S; ++s) {
        const NetShape& sh = shapes[s];
        OPB_REQUIRE(sh.hp % 8 == 0 && sh.wp % 8 == 0 && sh.n >= 1, "padded input dims must be multiples of 8");
        OPB_REQUIRE(sh.in_elem == 1 || sh.in_elem == 2, "net input is uint8 or bf16");
        TensorView in = B.act(sh.n, sh.hp, sh.wp, 3, sh.in_elem);
        plan->in_u8.push_back((uint8_t*)in.base);
        TensorView out = B.act(sh.n, sh.hp, sh.wp, 64);
        const DevLayer& d = net->dev.at("conv1_1");
        plan->steps.push_back([in, out, d](cudaStream_t st) { conv_first_launch(in, out, d.w_first, d.bias, st); });
        plan->step_names.push_back("conv_first:conv1_1");
        plan->step_gflop.push_back(B.add_flops("conv1_1", in));
        plan->kernel_launches += 1;
        StepInfo info;
        info.kind = kStepConvFirst;
        info.probs.push_back({"conv1_1", "", s, in, out});
        plan->step_info.push_back(info);
        cur[s] = out;
    }

    std::vector<int> scale_ids(S), branch_scale_ids(2 * S);
    for (int s = 0; s < S; ++s) scale_ids[s] = branch_scale_ids[2 * s] = branch_scale_ids[2 * s + 1] = s;

    // ---- VGG trunk on tensor cores, all scales grouped per layer ----
    auto trunk = [&](const std::string& name, int cout, bool pool, std::vector<TensorView>* into = nullptr) {
        std::vector<TensorView> outs(S);
        for (int s = 0; s < S; ++s) {
            if (into)
                outs[s] = (*into)[s];
            else if (pool && B.fuse_pool)
                outs[s] = B.act(cur[s].n, cur[s].h / 2, cur[s].w / 2, cout);
            else
                outs[s] = B.act(cur[s].n, cur[s].h, cur[s].w, cout);
        }
        B.conv_group(std::vector<std::string>(S, name), scale_ids, cur, outs, pool && B.fuse_pool);
        if (pool && !B.fuse_pool) {
            for (int s = 0; s < S; ++s) {
                TensorView pooled = B.act(outs[s].n, outs[s].h / 2, outs[s].w / 2, cout);
                TensorView full = outs[s];
                plan->steps.push_back([full, pooled](cudaStream_t st) { maxpool2_launch(full, pooled, st); });
                plan->step_names.push_back("maxpool2");
                plan->step_gflop.push_back(0.0);
                plan->kernel_launches += 1;
                StepInfo info;
                info.kind = kStepPool;
                info.probs.push_back({name, "", s, full, pooled});
                plan->step_info.push_back(info);
                outs[s] = pooled;
            }
        }
        cur = outs;
    };
    trunk("conv1_2", 64, true);
    trunk("conv2_1", 128, false);
    trunk("conv2_2", 128, true);
    trunk("conv3_1", 256, false);
    trunk("conv3_2", 256, false);
    trunk("conv3_3", 256, false);
    trunk("conv3_4", 256, true);
    trunk("conv4_1", 512, false);
    trunk("conv4_2", 512, false);

    // concat buffers (zero-filled once: pad channels must stay finite and zero)
    std::vector<TensorView> cat(S), feat(S);
    for (int s = 0; s < S; ++s) {
        cat[s] = B.act(cur[s].n, cur[s].h, cur[s].w, 192, 2, true);
        feat[s] = Builder::slice(cat[s], 0, 128);
    }
    char buf[64];
    if (body) {
        trunk("conv4_3_CPM", 256, false);
        trunk("conv4_4_CPM", 128, false, &feat);
        std::vector<TensorView> paf_slice(S), heat_slice(S);
        for (int s = 0; s < S; ++s) {
            paf_slice[s] = Builder::slice(cat[s], 128, 40);
            heat_slice[s] = Builder::slice(cat[s], 168, 24);
            TensorView op = B.act(cat[s].n, cat[s].h, cat[s].w, 40, 4, true);
            TensorView oh = B.act(cat[s].n, cat[s].h, cat[s].w, 24, 4, true);
            plan->out_paf.push_back((float*)op.base);
            plan->out_heat.push_back((float*)oh.base);
        }
        // per (scale, branch) ping-pong buffers
        std::vector<TensorView> pa(2 * S), pb(2 * S), wide(2 * S);
        for (int s = 0; s < S; ++s)
            for (int b = 0; b < 2; ++b) {
                pa[2 * s + b] = B.act(cat[s].n, cat[s].h, cat[s].w, 128);
                pb[2 * s + b] = B.act(cat[s].n, cat[s].h, cat[s].w, 128);
                wide[2 * s + b] = B.act(cat[s].n, cat[s].h, cat[s].w, 512);
            }
        auto branch_layer = [&](const char* fmt, int stage, const std::vector<TensorView>& ins,
                                const std::vector<TensorView>& outs, bool two_args) {
            std::vector<std::string> names(2 * S);
            for (int s = 0; s < S; ++s)
                for (int b = 0; b < 2; ++b) {
                    if (two_args) snprintf(buf, sizeof buf, fmt, stage, b + 1);
                    else snprintf(buf, sizeof buf, fmt, b + 1);
                    names[2 * s + b] = buf;
                }
            // problems of one launch must share block_n: group by branch when they differ
            std::vector<std::string> n1, n2;
            std::vector<TensorView> i1, i2, o1, o2;
            const int bn0 = net->dev.at(names[0]).block_n, bn1 = net->dev.at(names[1]).block_n;
            if (bn0 == bn1) {
                B.conv_group(names, branch_scale_ids, ins, outs, false);
            } else {
                for (int s = 0; s < S; ++s) {
                    n1.push_back(names[2 * s]); i1.push_back(ins[2 * s]); o1.push_back(outs[2 * s]);
                    n2.push_back(names[2 * s + 1]); i2.push_back(ins[2 * s + 1]); o2.push_back(outs[2 * s + 1]);
                }
                B.conv_group(n1, scale_ids, i1, o1, false);
                B.conv_group(n2, scale_ids, i2, o2, false);
            }
        };
        auto both = [&](const std::vector<TensorView>& per_scale) {
            std::vector<TensorView> v(2 * S);
            for (int s = 0; s < S; ++s) v[2 * s] = v[2 * s + 1] = per_scale[s];
            return v;
        };
        auto slices = [&](bool final_stage) {
            std::vector<TensorView> v(2 * S);
            for (int s = 0; s < S; ++s) {
                if (final_stage) {
                    TensorView op = cat[s];
                    op.base = plan->out_paf[s]; op.c = op.cstride = 40; op.coff = 0; op.elem = 4;
                    TensorView oh = cat[s];
                    oh.base = plan->out_heat[s]; oh.c = oh.cstride = 24; oh.coff = 0; oh.elem = 4;
                    v[2 * s] = op;
                    v[2 * s + 1] = oh;
                } else {
                    v[2 * s] = paf_slice[s];
                    v[2 * s + 1] = heat_slice[s];
                }
            }
            return v;
        };
        // stage 1 (src/model.py:52-62)
        branch_layer("conv5_1_CPM_L%d", 0, both(feat), pa, false);
        branch_layer("conv5_2_CPM_L%d", 0, pa, pb, false);
        branch_layer("conv5_3_CPM_L%d", 0, pb, pa, false);
        {
            std::vector<std::string> n4(2 * S), n5(2 * S);
            for (int s = 0; s < S; ++s)
                for (int b = 0; b < 2; ++b) {
                    snprintf(buf, sizeof buf, "conv5_4_CPM_L%d", b + 1);
                    n4[2 * s + b] = buf;
                    snprintf(buf, sizeof buf, "conv5_5_CPM_L%d", b + 1);
                    n5[2 * s + b] = buf;
                }
            if (!B.wide_tail_group(n4, n5, branch_scale_ids, pa, slices(false))) {
                branch_layer("conv5_4_CPM_L%d", 0, pa, wide, false);
                branch_layer("conv5_5_CPM_L%d", 0, wide, slices(false), false);
            }
        }
        // stages 2..6 (src/model.py:69-87)
        for (int st = 2; st <= 6; ++st) {
            branch_layer("Mconv1_stage%d_L%d", st, both(cat), pa, true);
            branch_layer("Mconv2_stage%d_L%d", st, pa, pb, true);
            branch_layer("Mconv3_stage%d_L%d", st, pb, pa, true);
            branch_layer("Mconv4_stage%d_L%d", st, pa, pb, true);
            branch_layer("Mconv5_stage%d_L%d", st, pb, pa, true);
            std::vector<std::string> n6(2 * S), n7(2 * S);
            for (int s = 0; s < S; ++s)
                for (int b = 0; b < 2; ++b) {
                    snprintf(buf, sizeof buf, "Mconv6_stage%d_L%d", st, b + 1);
                    n6[2 * s + b] = buf;
                    snprintf(buf, sizeof buf, "Mconv7_stage%d_L%d", st, b + 1);
                    n7[2 * s + b] = buf;
                }
            if (!B.tail_group(n6, n7, branch_scale_ids, pa, slices(st == 6))) {
                branch_layer("Mconv6_stage%d_L%d", st, pa, pb, true);
                branch_layer("Mconv7_stage%d_L%d", st, pb, slices(st == 6), true);
            }
        }
    } else {
        trunk("conv4_3", 512, false);
        trunk("conv4_4", 512, false);
        trunk("conv5_1", 512, false);
        trunk("conv5_2", 512, false);
        trunk("conv5_3_CPM", 128, false, &feat);
        std::vector<TensorView> heat_slice(S), final_out(S), pa(S), pb(S), wide(S);
        for (int s = 0; s < S; ++s) {
            heat_slice[s] = Builder::slice(cat[s], 128, 24);
            TensorView oh = B.act(cat[s].n, cat[s].h, cat[s].w, 24, 4, true);
            plan->out_heat.push_back((float*)oh.base);
            plan->out_paf.push_back(nullptr);
            final_out[s] = oh;
            pa[s] = B.act(cat[s].n, cat[s].h, cat[s].w, 128);
            pb[s] = B.act(cat[s].n, cat[s].h, cat[s].w, 128);
            wide[s] = B.act(cat[s].n, cat[s].h, cat[s].w, 512);
        }
        auto layer = [&](const std::string& name, const std::vector<TensorView>& ins, const std::vector<TensorView>& outs) {
            B.conv_group(std::vector<std::string>(S, name), scale_ids, ins, outs, false);
        };
        if (!B.wide_tail_group(std::vector<std::string>(S, "conv6_1_CPM"), std::vector<std::string>(S, "conv6_2_CPM"), scale_ids,
                               feat, heat_slice)) {
            layer("conv6_1_CPM", feat, wide);
            layer("conv6_2_CPM", wide, heat_slice);
        }
        for (int st = 2; st <= 6; ++st) {
            auto nm = [&](int i) {
                snprintf(buf, sizeof buf, "Mconv%d_stage%d", i, st);
                return std::string(buf);
            };
            layer(nm(1), cat, pa);
            layer(nm(2), pa, pb);
            layer(nm(3), pb, pa);
            layer(nm(4), pa, pb);
            layer(nm(5), pb, pa);
            if (!B.tail_group(std::vector<std::string>(S, nm(6)), std::vector<std::string>(S, nm(7)), scale_ids, pa,
                              st == 6 ? final_out : heat_slice)) {
                layer(nm(6), pa, pb);
                layer(nm(7), pb, st == 6 ? final_out : heat_slice);
            }
        }
    }
    OPB_REQUIRE(plan->step_info.size() == plan->steps.size(), "plan: step metadata out of step");
    return plan;
}

// ------------------------------------------------------------------------------------------------
// cubic tap tables (OpenCV semantics; oracle: cubic_taps / composite_upsample_matrix)
// ------------------------------------------------------------------------------------------------
int resize_dsize(int n, double f) { return (int)std::nearbyint((double)n * f); }   // default FE_TONEAREST = half-even

CubicTaps cubic_taps(int src, int dst, double scale) {
    (void)src;
    CubicTaps t;
    t.first.resize(dst);
    t.coef.resize((size_t)dst * 4);
    const float A = -0.75f;
    for (int d = 0; d < dst; ++d) {
        float fx = (float)((d + 0.5) * scale - 0.5);
        const int sx = (int)std::floor(fx);
        volatile float frac = fx - (float)sx;             // volatile: keep every float32 rounding (no x87/FMA games)
        const float x = frac;
        volatile float x1 = x + 1.0f;
        volatile float a0 = A * x1;
        volatile float a1 = a0 - 5.0f * A;
        volatile float a2 = a1 * x1;
        volatile float a3 = a2 + 8.0f * A;
        volatile float a4 = a3 * x1;
        const float c0 = a4 - 4.0f * A;
        volatile float b0 = (A + 2.0f) * x;
        volatile float b1 = b0 - (A + 3.0f);
        volatile float b2 = b1 * x;
        volatile float b3 = b2 * x;
        const float c1 = b3 + 1.0f;
        volatile float y = 1.0f - x;
        volatile float d0 = (A + 2.0f) * y;
        volatile float d1 = d0 - (A + 3.0f);
        volatile float d2 = d1 * y;
        volatile float d3 = d2 * y;
        const float c2 = d3 + 1.0f;
        volatile float e0 = 1.0f - c0;
        volatile float e1 = e0 - c1;
        const float c3 = e1 - c2;
        t.first[d] = sx - 1;
        t.coef[(size_t)d * 4 + 0] = c0;
        t.coef[(size_t)d * 4 + 1] = c1;
        t.coef[(size_t)d * 4 + 2] = c2;
        t.coef[(size_t)d * 4 + 3] = c3;
    }
    return t;
}

// composite 1-D operator: x8 cubic upsample of n_net samples -> crop to n_resized -> cubic resize to n_orig
void composite_taps(int n_net, int n_resized, int n_orig, std::vector<int>& first, std::vector<float>& w6) {
    const CubicTaps up = cubic_taps(n_net, n_net * 8, 1.0 / 8.0);
    const CubicTaps down = cubic_taps(n_resized, n_orig, 1.0 / ((double)n_orig / (double)n_resized));
    first.assign(n_orig, 0);
    w6.assign((size_t)n_orig * kUpTaps, 0.f);
    std::vector<double> acc(n_net);
    for (int o = 0; o < n_orig; ++o) {
        std::fill(acc.begin(), acc.end(), 0.0);
        int lo = n_net, hi = -1;
        for (int k = 0; k < 4; ++k) {
            int mid = down.first[o] + k;
            mid = mid < 0 ? 0 : (mid > n_resized - 1 ? n_resized - 1 : mid);       // clamped tap of pass 2
            const double dk = down.coef[(size_t)o * 4 + k];
            for (int l = 0; l < 4; ++l) {
                int sidx = up.first[mid] + l;
                sidx = sidx < 0 ? 0 : (sidx > n_net - 1 ? n_net - 1 : sidx);       // clamped tap of pass 1
                acc[sidx] += dk * (double)up.coef[(size_t)mid * 4 + l];
                lo = sidx < lo ? sidx : lo;
                hi = sidx > hi ? sidx : hi;
            }
        }
        if (hi - lo + 1 > kUpTaps)
            throw Error(OPB_ERR_INVALID, "composite cubic footprint wider than 6 taps (unsupported resize ratio)");
        first[o] = lo;
        for (int q = lo; q <= hi; ++q) w6[(size_t)o * kUpTaps + (q - lo)] = (float)acc[q];
    }
}

}  // namespace opb

opb_context::~opb_context() {
    for (void* p : owned) cudaFree(p);
    if (stream) cudaStreamDestroy(stream);
}
opb_net::~opb_net() {
    for (void* p : owned) cudaFree(p);
}
