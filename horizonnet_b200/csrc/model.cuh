// Internals of libhorizonnet_b200 shared by model.cu (inference schedule + C ABI) and train_step.cu (training step):
// the weight registry / graph / workspace object behind the opaque hn_model handle, and the helpers around it.
#pragma once
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "hn_common.cuh"
#include "conv_tc.cuh"

#define HN_NUM_CLASSES 8

namespace hn {

int ghc_to_sequence(const Act ghc[4], float* seq, cudaStream_t st, bool split);
int linear_head(const float* rnn, const float* w, const float* bias, float* bon, float* cor, int T, int B,
                cudaStream_t st);
int lstm_layer(const float* xproj, const float* w_hh_fwd, const float* w_hh_bwd, float* out, int T, int B,
               void* scratch, int* error_flag, cudaStream_t st);
size_t lstm_scratch_bytes();
int tta_views(const float* x, float* views, int B, int V, const int* modes_dev, const int* shifts_dev, cudaStream_t st);
int tta_merge(const float* bon, const float* cor, int B, int V, const int* modes_dev, const int* shifts_dev, float* y_bon,
              float* y_cor, cudaStream_t st);
size_t layout_workspace_bytes(int B);
int layout(const float* y_bon_pix, const float* y_cor, int B, int mode, float min_v, int r_px, void* workspace,
           float* cor_id, int* n_cor, float* z1, int* status, int* peaks, int* types, cudaStream_t st);
int pano_stretch_device(const float* img, float* out, int n, int H, int W, int C, const double* kx_dev,
                        const double* ky_dev, double* scratch, int order, cudaStream_t st);
int pano_stretch_device_f64(const double* img, double* out, int n, int H, int W, int C, const double* kx_dev,
                            const double* ky_dev, double* scratch, int order, cudaStream_t st);
int augment_device(const unsigned char* img, float* out, int n, int H, int W, const double* kx_dev, const double* ky_dev,
                   const int* params_dev, double* scratch, cudaStream_t st);
int rotate_panorama_device(const void* img, int in_f64, double* out, int n, int H, int W, int C, const double* rinv,
                           cudaStream_t st);



// Entry points run on the model's device and restore the caller's current device on return (a multi-GPU
// single-process caller must not find its current device switched by a forward on another GPU).
struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) ok = (cudaSetDevice(dev) == cudaSuccess);
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
#define HN_ON_DEVICE(dev)                                                                  \
    DeviceGuard _dg(dev);                                                                  \
    if (!_dg.ok) return ::hn::fail("cudaSetDevice failed for the model's device")


enum { CLS_STEM = 0, CLS_POOL, CLS_ENC_CONV, CLS_GHC_CONV, CLS_TAIL, CLS_XPROJ, CLS_LSTM, CLS_HEAD };

struct TensorSlot {
    std::string key;
    long long numel = 0;
    float* dev = nullptr;     // staging copy in the reference layout
    bool set = false;
    bool ignored = false;     // num_batches_tracked
};

struct ConvLayer {
    ConvDesc d;
    std::string wkey, bnprefix, biaskey;
    float* w = nullptr;
    float* scale = nullptr;
    float* shift = nullptr;
    unsigned short* wq = nullptr;     // [2][Cout][K] hi/lo weight planes for the tcgen05 kernel
    float* tc_scale = nullptr;        // 3*Cout (+1 scratch) epilogue constants of the tcgen05 path (conv_tc.cuh: tc_aux)
    int bn_index = -1;                // position in hn_model::bn_names (train mode: which BatchNorm2d module this is)
};

// Train-mode forward (hn_model_forward_train): per-BatchNorm2d switches handed in by the caller
struct TrainCtx {
    const unsigned char* bn_train;    // [n_bn] 1: batch statistics + running update, 0: module is in eval mode
    const double* bn_factor;          // [n_bn] exponential_average_factor (momentum, or 1/num_batches_tracked); < 0: none
    unsigned long long seed;
    double rnn_p, head_p;             // dropout probabilities (0: off)
    const float* mask[2];             // caller-supplied multiplicative masks instead of the Philox ones (parity tests)
};


}  // namespace hn

using namespace hn;       // every includer is an implementation file of this library

struct hn_model {
    int device = 0;
    int max_batch = 0;
    bool finalized = false;
    int use_tc = 0;                                  // 1: route supported convs through tcgen05 kernels
    std::vector<TensorSlot> slots;
    std::map<std::string, int> index;
    std::vector<void*> allocs;

    // graph
    ConvLayer stem;                                  // weights packed [147][64]
    unsigned short* stem_wq = nullptr;               // tcgen05 stem: [2][64][224] fp16 planes (conv_tc.cu: stem_tc)
    float* stem_aux = nullptr;                       // 3*64 + 1 epilogue constants
    int stem_tc_on = 1;                              // option "stem_tc" / HN_TC_STEM=0: fp32 CUDA-core stem inside the TC path
    int fuse_on = 1;                                 // option "fuse_bottleneck": fused conv2+conv3 kernel for layer1 (bit-identical)
    struct Block { ConvLayer c1, c2, c3, ds; bool has_ds = false; };
    std::vector<Block> blocks[4];
    ConvLayer ghc[4][4];
    ConvLayer xproj[2];                              // LSTM input projections as 1x1 convs, N = 4096
    float* head_w = nullptr;
    float* head_b = nullptr;
    const float* whh[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};
    std::vector<std::string> bn_names;               // state_dict prefixes of the 69 BatchNorm2d modules, graph order
    // train-mode scratch (one layer at a time, stream ordered): batch sums, scale/shift, tcgen05 epilogue constants
    std::shared_ptr<void> train_state;               // tape + gradient buffers of the training step (train_step.cu)
    bool bn_stale = false;     // running statistics moved (train forward) since the eval-mode constants were folded
    double* trn_sums = nullptr;
    float *trn_scale = nullptr, *trn_shift = nullptr, *trn_aux = nullptr;

    // workspace (sized for max_batch)
    float *S0 = nullptr, *S1 = nullptr, *X[2] = {nullptr, nullptr}, *IDN = nullptr, *T1 = nullptr, *T2 = nullptr;
    float* F[4] = {nullptr, nullptr, nullptr, nullptr};
    float* G[2] = {nullptr, nullptr};
    float* GO[4] = {nullptr, nullptr, nullptr, nullptr};
    float *SEQ = nullptr, *XP = nullptr, *R1 = nullptr, *R2 = nullptr, *R1S = nullptr;
    unsigned int* counters = nullptr;
    int* error_flag = nullptr;
    float *x_in = nullptr, *bon_out = nullptr, *cor_out = nullptr;    // for forward_host
    // pipelined host API: 2 input slots, a copy stream and a compute stream (H2D of batch i+1 overlaps forward i)
    float* x_slot[2] = {nullptr, nullptr};
    cudaStream_t copy_stream = nullptr, compute_stream = nullptr;
    cudaEvent_t slot_ready[2] = {nullptr, nullptr};
    int slot_batch[2] = {0, 0};
    int submit_count = 0, collect_count = 0;
    float* bon_slot[2] = {nullptr, nullptr};        // device outputs of the two host-pipeline slots
    float* cor_slot[2] = {nullptr, nullptr};
    // Two-stream schedule of the throughput entry points (hn_model_forward_async, submit/collect): the encoder +
    // height reduction of batch i+1 run on enc_stream while the bi-LSTM + head of batch i (64 of the 148 SMs,
    // latency-bound) run on the high-priority rnn_stream.
    cudaStream_t enc_stream = nullptr, rnn_stream = nullptr;
    cudaEvent_t ev_in = nullptr, ev_xfree = nullptr, ev_seq = nullptr, ev_rnn_last = nullptr, ev_plain_done = nullptr;
    cudaEvent_t async_done[2] = {nullptr, nullptr}, slot_done[2] = {nullptr, nullptr};
    bool rnn_inflight = false, plain_recorded = false;
    long long async_count = 0;
    int* tta_ints = nullptr;                        // [2][64] view modes / shifts for hn_model_infer_tta
    int last_batch = 0;

    // optional per-op-class timing (bench.py roofline): CUDA event pairs around every launch
    int profile = 0;
    struct Span { int cls; double flops; cudaEvent_t a, b; };
    std::vector<Span> spans;                       // pending (recorded, not yet read)
    std::vector<cudaEvent_t> free_events;
    double prof_ms[HN_NUM_CLASSES] = {0};
    double prof_flops[HN_NUM_CLASSES] = {0};
    long long prof_launches[HN_NUM_CLASSES] = {0};

    ~hn_model() {
        int prev_dev = -1;
        if (cudaGetDevice(&prev_dev) != cudaSuccess) prev_dev = -1;
        cudaSetDevice(device);
        for (auto& sp : spans) { cudaEventDestroy(sp.a); cudaEventDestroy(sp.b); }
        for (auto e : free_events) cudaEventDestroy(e);
        for (int i = 0; i < 2; ++i) if (slot_ready[i]) cudaEventDestroy(slot_ready[i]);
        if (copy_stream) cudaStreamDestroy(copy_stream);
        if (compute_stream) cudaStreamDestroy(compute_stream);
        for (cudaEvent_t e : {ev_in, ev_xfree, ev_seq, ev_rnn_last, ev_plain_done, async_done[0], async_done[1],
                              slot_done[0], slot_done[1]})
            if (e) cudaEventDestroy(e);
        if (enc_stream) cudaStreamDestroy(enc_stream);
        if (rnn_stream) cudaStreamDestroy(rnn_stream);
        for (void* p : allocs) cudaFree(p);
        if (prev_dev >= 0) cudaSetDevice(prev_dev);
    }
    cudaEvent_t get_event() {
        if (!free_events.empty()) { cudaEvent_t e = free_events.back(); free_events.pop_back(); return e; }
        cudaEvent_t e; cudaEventCreate(&e); return e;
    }
    int alloc(void** p, size_t bytes) {
        HN_CUDA_OK(cudaMalloc(p, bytes ? bytes : 4));
        allocs.push_back(*p);
        return 0;
    }
    template <typename T>
    int alloc_t(T** p, size_t n) { return alloc(reinterpret_cast<void**>(p), n * sizeof(T)); }

    int add_slot(const std::string& key, long long numel, bool ignored = false) {
        TensorSlot s;
        s.key = key; s.numel = numel; s.ignored = ignored;
        index[key] = (int)slots.size();
        slots.push_back(s);
        return 0;
    }
    void add_bn(const std::string& p, int c) {
        add_slot(p + ".weight", c); add_slot(p + ".bias", c);
        add_slot(p + ".running_mean", c); add_slot(p + ".running_var", c);
        add_slot(p + ".num_batches_tracked", 1, true);
    }
    const float* T(const std::string& key) const { return slots[index.at(key)].dev; }
};

namespace hn {

inline Act mk(float* p, int B, int H, int W, int C, int halo = 1) {
    Act a; a.p = p; a.B = B; a.H = H; a.W = W; a.C = C; a.halo = halo; return a;
}

// RAII span: records an event pair around the launches issued in its scope when profiling is on
struct Scope {
    hn_model* m; cudaStream_t st; hn_model::Span sp; bool on;
    Scope(hn_model* m_, int cls, double flops, cudaStream_t st_) : m(m_), st(st_), on(m_->profile != 0) {
        if (!on) return;
        sp.cls = cls; sp.flops = flops; sp.a = m->get_event(); sp.b = m->get_event();
        cudaEventRecord(sp.a, st);
    }
    ~Scope() {
        if (!on) return;
        cudaEventRecord(sp.b, st);
        m->spans.push_back(sp);
    }
};

}  // namespace hn
