// Host-side runtime of the library: contexts, network weights, execution plans, sessions.
#pragma once
#include "opb_common.cuh"
#include <functional>
#include <memory>

namespace opb {

struct LayerSpec {
    std::string name;
    int cin, cout, k;
    bool relu;
    bool pool_after;      // a 2x2/2 max-pool follows this layer (src/model.py:37,40,45)
};
const std::vector<LayerSpec>& layer_specs(int kind);

// device weights of one layer in the layout the kernels consume
struct DevLayer {
    __nv_bfloat16* w = nullptr;   // [cout_pad][k*k*cin_dev] bf16 (tensor-core layers)
    float* w_first = nullptr;     // [27][64] fp32 holding bf16-rounded values (conv1_1 only)
    float* bias = nullptr;        // [cout_pad] fp32
    __nv_bfloat16* w_wide = nullptr;   // 64 -> 64 channel 3x3 layers (conv1_2): [128][9 * 128] wide-pixel weights (wide_pool_weights)
    float* bias_wide = nullptr;        // [128]: the bias twice
    int cin_dev = 0;              // channels of the device input view (padded / permuted)
    int cout_pad = 0, cout_store = 0, block_n = 128, k = 3;
    bool relu = true;
};

struct HostLayer {
    std::vector<float> w, b;
    int cout = 0, cin = 0, k = 0;
};

}  // namespace opb

struct opb_context {
    int device = 0;
    cudaStream_t stream = nullptr;
    int num_sms = 148;
    int64_t launches = 0;
    // scratch for the stage-level entry points
    std::vector<void*> owned;
    ~opb_context();
};

struct opb_net {
    opb_context* ctx = nullptr;
    int kind = OPB_NET_BODY;
    std::map<std::string, opb::HostLayer> host;
    std::map<std::string, opb::DevLayer> dev;
    bool finalized = false;
    std::vector<void*> owned;
    // sessions keep their network alive: opb_net_destroy on a net that still has sessions only marks it, the last
    // opb_session_destroy frees it (a garbage collector may finalise the two host objects in either order)
    int sessions = 0;
    bool released = false;
    ~opb_net();
};

namespace opb {

// a device allocation list freed with its owner
struct DevPool {
    std::vector<void*> ptrs;
    size_t bytes = 0;
    void* alloc(size_t n, bool zero = false);
    template <typename T>
    T* alloc_t(size_t count, bool zero = false) { return (T*)alloc(count * sizeof(T), zero); }
    template <typename T>
    T* upload(const std::vector<T>& v) {
        T* d = alloc_t<T>(v.size() ? v.size() : 1);
        if (!v.empty()) OPB_CUDA(cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
        return d;
    }
    void release();
    ~DevPool() { release(); }
};

// CNN execution plan for a fixed set of input shapes (one entry per scale)
struct NetShape {
    int n, hp, wp;
    int in_elem = 1;          // bytes per input element: 1 = uint8 pixels, 2 = bf16 (batched estimators' float frames)
    bool operator<(const NetShape& o) const {
        if (n != o.n) return n < o.n;
        if (hp != o.hp) return hp < o.hp;
        if (wp != o.wp) return wp < o.wp;
        return in_elem < o.in_elem;
    }
};
// per-step CUDA-event profiler (bench.py roofline numbers; off by default)
struct Profiler {
    bool on = false;
    std::vector<cudaEvent_t> ev;
    std::vector<std::string> names;
    std::vector<double> gflop;
    size_t used = 0;
    void reset() { used = 0; names.clear(); gflop.clear(); }
    void mark(cudaStream_t st, const std::string& name, double gf = 0.0) {
        if (!on) return;
        if (used == ev.size()) {
            cudaEvent_t e;
            OPB_CUDA(cudaEventCreate(&e));
            ev.push_back(e);
        }
        OPB_CUDA(cudaEventRecord(ev[used++], st));
        names.push_back(name);
        gflop.push_back(gf);
    }
    ~Profiler() {
        for (auto e : ev) cudaEventDestroy(e);
    }
};

// What one step of a plan computes, for the layer-by-layer tests (opb_net_debug_*): host metadata only.
enum StepKind {
    kStepConvFirst = OPB_STEP_CONV_FIRST, kStepConv = OPB_STEP_CONV, kStepTail = OPB_STEP_TAIL,
    kStepTailWide = OPB_STEP_TAIL_WIDE, kStepPool = OPB_STEP_POOL
};
struct StepProblem {
    std::string layer, layer2;      // layer2: the second layer of a fused tail
    int scale = 0;                  // index into NetPlan::shapes
    TensorView in, out;             // conv1_2 in its wide-pixel form: the views of the plain layer
};
struct StepInfo {
    int kind = kStepConv;
    std::vector<StepProblem> probs;
    int block_n = 0;                // N tile of a tensor-core launch
    bool pool = false;              // fused 2x2 max-pool
    bool wide = false;              // conv1_2 ran in the wide-pixel form
    bool pair = false;              // CTA-pair kernel
    bool half_tiles = false;        // CTA pair: 16 x 8 tiles
    bool weights_resident = false;  // CTA pair: the weight set stays in shared memory (bres)
};

struct NetPlan {
    DevPool pool;
    std::vector<NetShape> shapes;
    std::vector<uint8_t*> in_u8;                // per scale: (n, hp, wp, 3) uint8 (or bf16, NetShape::in_elem) input
    std::vector<float*> out_paf, out_heat;      // per scale: fp32 NHWC (cstride 40 / 24); hand: heat only
    std::vector<std::function<void(cudaStream_t)>> steps;
    std::vector<std::string> step_names;        // parallel to steps
    std::vector<StepInfo> step_info;            // parallel to steps
    std::vector<double> step_gflop;
    std::vector<ConvLaunch*> launches;
    int kernel_launches = 0;
    double gflop = 0;                           // algorithmic FLOPs (un-padded channels), for the roofline
    void run(cudaStream_t s, Profiler* prof = nullptr) const {
        for (size_t i = 0; i < steps.size(); ++i) {
            steps[i](s);
            if (prof) prof->mark(s, step_names[i], step_gflop[i]);
        }
    }
    ~NetPlan();
};
std::unique_ptr<NetPlan> build_net_plan(opb_net* net, const std::vector<NetShape>& shapes);
void finalize_net(opb_net* net);
constexpr int kDefaultConvImpl = 2;       // measured on B200 (bench.py, 720p 4-scale, same box): CTA pair 3.60 ms of conv per frame, patch MODE 1 3.79, MODE 0 and per-tap slower
int default_conv_impl();
// Wide-pixel form of a 64 -> 64 channel 3x3 layer + 2x2 pool (ConvOp::pool_wide).  weight: [64][64][9] fp32 (cout, cin, tap).
void wide_pool_weights(const float* weight, const float* bias, std::vector<__nv_bfloat16>& w_wide, std::vector<float>& b_wide);
// `base`: the layer as a plain pooled problem (in (n, h, w, 64) contiguous, out (n, h/2, w/2, 64)); w even.
ConvOp wide_pool_op(const ConvOp& base, const __nv_bfloat16* w_wide, const float* b_wide);
bool wide_pool_ok(const ConvOp& base);

// cubic tap tables (host)
struct CubicTaps {
    std::vector<int> first;       // first source index (unclamped), per destination index
    std::vector<float> coef;      // [dst][4] float32 coefficients
};
CubicTaps cubic_taps(int src, int dst, double scale);
// torch's bicubic taps; scale_factor <= 0: size mode (dst given, step float(src) / float(dst))
CubicTaps torch_cubic_taps(int src, int dst, double scale_factor);
int resize_dsize(int n, double f);                 // cv2: saturate_cast<int>(n*f), round half to even
void composite_taps(int n_net, int n_resized, int n_orig, std::vector<int>& first, std::vector<float>& w6,
                    bool torch = false);

}  // namespace opb
