// hn_model: weight registry (reference checkpoint layout, misc/utils.py:49-65), BN folding and
// weight packing, activation workspace, and the forward schedule of HorizonNet('resnet50', rnn)
// (reference model.py:254-281), plus the C ABI (include/horizonnet_b200.h).
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>
#include <atomic>

#include "model.cuh"
#include "../../include/horizonnet_b200.h"

#ifndef HN_BUILD_DIGEST
#define HN_BUILD_DIGEST "unknown"
#endif

namespace hn {

// ---- error / launch accounting -----------------------------------------------------------------
static thread_local std::string g_err;
static std::atomic<long long> g_launches{0};
void set_error(const std::string& m) { g_err = m; }
int fail(const std::string& m) { g_err = m; return -1; }
void count_launch(int n) { g_launches += n; }

namespace {
// ---- packing kernels ---------------------------------------------------------------------------
// OIHW [Cout][Cin][kh][kw] -> [K = (dy*kw+dx)*Cin + c][Cout]
__global__ void pack_oihw_kernel(const float* __restrict__ w, float* __restrict__ out, int Cout, int Cin, int kh,
                                 int kw) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t total = (size_t)Cout * Cin * kh * kw;
    if (i >= total) return;
    const int n = (int)(i % Cout);
    const size_t k = i / Cout;
    const int c = (int)(k % Cin);
    const int tap = (int)(k / Cin);
    const int dy = tap / kw, dx = tap % kw;
    out[i] = w[(((size_t)n * Cin + c) * kh + dy) * kw + dx];
}

// eval-mode BN (+ optional conv bias) -> scale/shift:  y = conv*scale + shift
__global__ void fold_bn_kernel(const float* __restrict__ gamma, const float* __restrict__ beta,
                               const float* __restrict__ mean, const float* __restrict__ var,
                               const float* __restrict__ bias, float* __restrict__ scale,
                               float* __restrict__ shift, int C) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= C) return;
    const double s = (double)gamma[i] / sqrt((double)var[i] + 1e-5);      // BatchNorm2d eps (model.py:130)
    const double b = bias ? (double)bias[i] : 0.0;
    scale[i] = (float)s;
    shift[i] = (float)((double)beta[i] + (b - (double)mean[i]) * s);
}

__global__ void lstm_bias_kernel(const float* __restrict__ bih_f, const float* __restrict__ bhh_f,
                                 const float* __restrict__ bih_b, const float* __restrict__ bhh_b,
                                 float* __restrict__ scale, float* __restrict__ shift) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 4096) return;
    scale[i] = 1.f;
    shift[i] = i < 2048 ? bih_f[i] + bhh_f[i] : bih_b[i - 2048] + bhh_b[i - 2048];
}

// halo-NHWC interior -> NCHW (test hook)
__global__ void nhwc_to_nchw_kernel(const float* __restrict__ in, float* __restrict__ out, int B, int H, int W,
                                    int C, int halo) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t total = (size_t)B * C * H * W;
    if (i >= total) return;
    const int w = (int)(i % W);
    size_t t = i / W;
    const int h = (int)(t % H); t /= H;
    const int c = (int)(t % C);
    const int b = (int)(t / C);
    out[i] = in[(((size_t)b * H + h) * (W + 2 * halo) + w + halo) * C + c];
}

// seq [T][B][1024] -> feature [B][1024][T]
__global__ void seq_to_feature_kernel(const float* __restrict__ seq, float* __restrict__ out, int T, int B) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t total = (size_t)T * B * 1024;
    if (i >= total) return;
    const int t = (int)(i % T);
    const int ch = (int)((i / T) % 1024);
    const int b = (int)(i / T / 1024);
    out[i] = seq[((size_t)t * B + b) * 1024 + ch];
}

}  // namespace
}  // namespace hn

using namespace hn;


namespace {

ConvLayer make_conv(hn_model* m, const std::string& wkey, const std::string& bn, const std::string& biaskey, int cin,
                    int cout, int k, int sh, int sw, int relu) {
    ConvLayer c;
    c.d.Cin = cin; c.d.Cout = cout; c.d.kh = k; c.d.kw = k; c.d.sh = sh; c.d.sw = sw;
    c.d.ph = k / 2; c.d.pw = k / 2; c.d.relu = relu;
    c.wkey = wkey; c.bnprefix = bn; c.biaskey = biaskey;
    m->add_slot(wkey, (long long)cout * cin * k * k);
    if (!biaskey.empty()) m->add_slot(biaskey, cout);
    m->add_bn(bn, cout);
    c.bn_index = (int)m->bn_names.size();
    m->bn_names.push_back(bn);
    return c;
}

// Builds the key list in the reference's own order (tests/golden/state_dict_keys.json) and the graph.
void build_graph(hn_model* m) {
    const std::string enc = "feature_extractor.encoder.";
    m->stem = make_conv(m, enc + "conv1.1.weight", enc + "bn1", "", 3, 64, 7, 2, 2, 1);
    const int nblk[4] = {3, 4, 6, 3};
    const int planes[4] = {64, 128, 256, 512};
    int inpl = 64;
    for (int l = 0; l < 4; ++l) {
        for (int b = 0; b < nblk[l]; ++b) {
            const std::string p = enc + "layer" + std::to_string(l + 1) + "." + std::to_string(b) + ".";
            const int stride = (b == 0 && l > 0) ? 2 : 1;
            hn_model::Block blk;
            blk.c1 = make_conv(m, p + "conv1.weight", p + "bn1", "", inpl, planes[l], 1, 1, 1, 1);
            blk.c2 = make_conv(m, p + "conv2.1.weight", p + "bn2", "", planes[l], planes[l], 3, stride, stride, 1);
            blk.c3 = make_conv(m, p + "conv3.weight", p + "bn3", "", planes[l], planes[l] * 4, 1, 1, 1, 1);
            blk.has_ds = (b == 0);
            if (blk.has_ds)
                blk.ds = make_conv(m, p + "downsample.0.weight", p + "downsample.1", "", inpl, planes[l] * 4, 1, stride,
                                   stride, 0);
            inpl = planes[l] * 4;
            m->blocks[l].push_back(blk);
        }
    }
    for (int s = 0; s < 4; ++s) {
        const int c = planes[s] * 4;
        const int ch[5] = {c, c / 2, c / 2, c / 4, c / 8};
        for (int j = 0; j < 4; ++j) {
            const std::string p =
                "reduce_height_module.ghc_lst." + std::to_string(s) + ".layer." + std::to_string(j) + ".layers.";
            m->ghc[s][j] = make_conv(m, p + "0.1.weight", p + "1", p + "0.1.bias", ch[j], ch[j + 1], 3, 2, 1, 1);
        }
    }
    for (int layer = 0; layer < 2; ++layer)
        for (int dir = 0; dir < 2; ++dir) {
            const std::string sfx = "_l" + std::to_string(layer) + (dir ? "_reverse" : "");
            m->add_slot("bi_rnn.weight_ih" + sfx, 2048ll * 1024);
            m->add_slot("bi_rnn.weight_hh" + sfx, 2048ll * 512);
            m->add_slot("bi_rnn.bias_ih" + sfx, 2048);
            m->add_slot("bi_rnn.bias_hh" + sfx, 2048);
        }
    m->add_slot("linear.weight", 12 * 1024);
    m->add_slot("linear.bias", 12);
    for (int layer = 0; layer < 2; ++layer) {
        ConvLayer& c = m->xproj[layer];
        c.d.Cin = 1024; c.d.Cout = 4096; c.d.kh = c.d.kw = 1; c.d.sh = c.d.sw = 1; c.d.ph = c.d.pw = 0; c.d.relu = 0;
    }
}

int pack_conv(hn_model* m, ConvLayer& c, cudaStream_t st) {
    const size_t nw = (size_t)c.d.Cout * c.d.Cin * c.d.kh * c.d.kw;
    if (!c.w) {
        if (m->alloc_t(&c.w, nw)) return -1;
        if (m->alloc_t(&c.scale, c.d.Cout)) return -1;
        if (m->alloc_t(&c.shift, c.d.Cout)) return -1;
        if (c.d.Cin % 64 == 0 && (m->alloc_t(&c.wq, 2 * nw) || m->alloc_t(&c.tc_scale, 3 * c.d.Cout + 1))) return -1;
    }
    pack_oihw_kernel<<<(unsigned)((nw + 255) / 256), 256, 0, st>>>(m->T(c.wkey), c.w, c.d.Cout, c.d.Cin, c.d.kh, c.d.kw);
    HN_LAUNCH_OK();
    fold_bn_kernel<<<(c.d.Cout + 255) / 256, 256, 0, st>>>(
        m->T(c.bnprefix + ".weight"), m->T(c.bnprefix + ".bias"), m->T(c.bnprefix + ".running_mean"),
        m->T(c.bnprefix + ".running_var"), c.biaskey.empty() ? nullptr : m->T(c.biaskey), c.scale, c.shift, c.d.Cout);
    HN_LAUNCH_OK();
    if (c.wq && pack_weight_tc(m->T(c.wkey), c.wq, c.scale, c.shift, c.tc_scale, c.tc_scale + 3 * c.d.Cout, c.d.Cout,
                               c.d.Cin, c.d.kh, c.d.kw, st))
        return -1;
    c.d.w = c.w; c.d.scale = c.scale; c.d.shift = c.shift;
    return 0;
}



int run_conv(hn_model* m, const ConvLayer& c, const Act& in, const Act& out, const float* res, cudaStream_t st,
             int cls, bool out_f32 = false) {
    const double flops = 2.0 * (double)out.B * out.H * out.W * c.d.Cout * c.d.kh * c.d.kw * c.d.Cin;
    Scope sc(m, cls, flops, st);
    if (!m->use_tc) return conv_f32(c.d, in, out, res, st);
    // tensor-core path: every activation buffer holds fp16 hi/lo planes (same bytes as fp32)
    if (!c.wq || !conv_tc_supported(c.d, in, out))
        return fail("hn_model_forward: a convolution of the graph is not covered by the tcgen05 kernel");
    return conv_tc_planes(c.d, c.wq, c.tc_scale, in, reinterpret_cast<const unsigned short*>(in.p), out,
                          out_f32 ? nullptr : reinterpret_cast<unsigned short*>(out.p), out_f32 ? out.p : nullptr,
                          reinterpret_cast<const unsigned short*>(res), st);
}

// Eval-mode epilogue constants again from the (moved) running statistics; the packed weights are untouched.
int refold_bn(hn_model* m, cudaStream_t st) {
    std::vector<ConvLayer*> all{&m->stem};
    for (int l = 0; l < 4; ++l)
        for (auto& b : m->blocks[l]) {
            all.push_back(&b.c1); all.push_back(&b.c2); all.push_back(&b.c3);
            if (b.has_ds) all.push_back(&b.ds);
        }
    for (int s = 0; s < 4; ++s)
        for (int j = 0; j < 4; ++j) all.push_back(&m->ghc[s][j]);
    for (ConvLayer* c : all) {
        const int C = c->d.Cout;
        fold_bn_kernel<<<(C + 255) / 256, 256, 0, st>>>(
            m->T(c->bnprefix + ".weight"), m->T(c->bnprefix + ".bias"), m->T(c->bnprefix + ".running_mean"),
            m->T(c->bnprefix + ".running_var"), c->biaskey.empty() ? nullptr : m->T(c->biaskey), c->scale, c->shift, C);
        HN_LAUNCH_OK();
        if (c->tc_scale && tc_aux_update(c->scale, c->shift, c->tc_scale + 3 * C, c->tc_scale, C, st)) return -1;
    }
    if (tc_aux_update(m->stem.scale, m->stem.shift, m->stem_aux + 3 * 64, m->stem_aux, 64, st)) return -1;
    m->bn_stale = false;
    return 0;
}

// conv + BatchNorm2d (+ identity, ReLU).  Eval (tr == nullptr, or a BN module the caller keeps in eval mode --
// train.py:251-256 --freeze_earlier_blocks): one launch with the running statistics folded into the epilogue.
// Train: the same convolution kernel twice -- raw output (+ conv bias) -> batch mean / biased variance and the
// running-statistics update (train_fwd.cu) -> the real pass with the batch statistics folded into the epilogue.
int conv_bn(hn_model* m, const ConvLayer& c, const Act& in, const Act& out, const float* res, cudaStream_t st, int cls,
            const TrainCtx* tr) {
    if (!tr || !tr->bn_train[c.bn_index]) return run_conv(m, c, in, out, res, st, cls);
    const int C = c.d.Cout;
    const float* bias = c.biaskey.empty() ? nullptr : m->T(c.biaskey);
    ConvLayer t = c;
    t.d.relu = 0; t.d.scale = m->trn_scale; t.d.shift = m->trn_shift; t.tc_scale = m->trn_aux;
    if (bn_identity_constants(bias, m->trn_scale, m->trn_shift, C, st)) return -1;
    if (m->use_tc && tc_aux_update(m->trn_scale, m->trn_shift, c.tc_scale + 3 * C, m->trn_aux, C, st)) return -1;
    if (run_conv(m, t, in, out, nullptr, st, cls)) return -1;
    if (bn_batch_stats(out, m->use_tc != 0, m->trn_sums, st)) return -1;
    if (bn_train_finalize(m->trn_sums, (long long)out.B * out.H * out.W, m->T(c.bnprefix + ".weight"),
                          m->T(c.bnprefix + ".bias"), bias, const_cast<float*>(m->T(c.bnprefix + ".running_mean")),
                          const_cast<float*>(m->T(c.bnprefix + ".running_var")), tr->bn_factor[c.bn_index],
                          m->trn_scale, m->trn_shift, C, st))
        return -1;
    if (m->use_tc && tc_aux_update(m->trn_scale, m->trn_shift, c.tc_scale + 3 * C, m->trn_aux, C, st)) return -1;
    t.d.relu = c.d.relu;
    return run_conv(m, t, in, out, res, st, cls);
}

}  // namespace

// ------------------------------------------------------------------------------------------------
extern "C" {

const char* hn_last_error(void) { return g_err.c_str(); }
int hn_abi_version(void) { return 2; }
const char* hn_build_digest(void) { return HN_BUILD_DIGEST; }
long long hn_kernel_launches(void) { return g_launches.load(); }

int hn_model_create(int device, int max_batch, hn_model** out) {
    HN_CHECK(out != nullptr, "hn_model_create: out is NULL");
    HN_CHECK(max_batch >= 1 && max_batch <= 1024, "hn_model_create: max_batch must be in 1..1024");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail("hn_model_create: no CUDA device -- libhorizonnet_b200 has no CPU path");
    HN_CHECK(device >= 0 && device < ndev, "hn_model_create: bad device index");
    HN_ON_DEVICE(device);
    cudaDeviceProp prop;
    HN_CUDA_OK(cudaGetDeviceProperties(&prop, device));
    HN_CHECK(prop.major == 10, "hn_model_create: this library is built for sm_100a (B200) only");
    std::unique_ptr<hn_model> m(new hn_model());
    m->device = device;
    m->max_batch = max_batch;
    if (const char* e = getenv("HN_TC_STEM")) m->stem_tc_on = atoi(e);
    build_graph(m.get());
    for (auto& s : m->slots)
        if (!s.ignored && m->alloc_t(&s.dev, (size_t)s.numel)) return -1;
    const size_t B = (size_t)max_batch;
    struct { float** p; size_t n; } bufs[] = {
        {&m->S0, B * 256 * 514 * 64},   {&m->S1, B * 128 * 258 * 64},  {&m->X[0], B * 128 * 258 * 256},
        {&m->X[1], B * 128 * 258 * 256}, {&m->IDN, B * 128 * 258 * 256}, {&m->T1, B * 128 * 258 * 128},
        {&m->T2, B * 128 * 258 * 64},   {&m->F[0], B * 128 * 258 * 256}, {&m->F[1], B * 64 * 130 * 512},
        {&m->F[2], B * 32 * 66 * 1024}, {&m->F[3], B * 16 * 34 * 2048}, {&m->G[0], B * 64 * 258 * 128},
        {&m->G[1], B * 64 * 258 * 128}, {&m->GO[0], B * 8 * 258 * 32},  {&m->GO[1], B * 4 * 130 * 64},
        {&m->GO[2], B * 2 * 66 * 128},  {&m->GO[3], B * 1 * 34 * 256},  {&m->SEQ, 256 * B * 1024},
        {&m->XP, (256 * B * 4096 > (size_t)4096 * 1024) ? 256 * B * 4096 : (size_t)4096 * 1024},       {&m->R1, 256 * B * 1024},       {&m->R2, 256 * B * 1024},       {&m->R1S, 256 * B * 1024},
        {&m->x_in, B * 3 * 512 * 1024}, {&m->bon_out, B * 2 * 1024},    {&m->cor_out, B * 1024},
        {&m->x_slot[1], B * 3 * 512 * 1024},
        {&m->bon_slot[1], B * 2 * 1024},  {&m->cor_slot[1], B * 1024},
        {&m->head_w, 12 * 1024},        {&m->head_b, 12},
    };
    for (auto& b : bufs)
        if (m->alloc_t(b.p, b.n)) return -1;
    if (m->alloc(reinterpret_cast<void**>(&m->counters), lstm_scratch_bytes())) return -1;
    if (m->alloc_t(&m->error_flag, 1)) return -1;
    if (m->alloc_t(&m->tta_ints, 128)) return -1;
    if (m->alloc_t(&m->trn_sums, 2 * 4096) || m->alloc_t(&m->trn_scale, 4096) || m->alloc_t(&m->trn_shift, 4096) ||
        m->alloc_t(&m->trn_aux, 3 * 4096 + 1))
        return -1;
    HN_CUDA_OK(cudaMemset(m->error_flag, 0, sizeof(int)));
    m->x_slot[0] = m->x_in;
    m->bon_slot[0] = m->bon_out; m->cor_slot[0] = m->cor_out;
    HN_CUDA_OK(cudaStreamCreateWithFlags(&m->copy_stream, cudaStreamNonBlocking));
    HN_CUDA_OK(cudaStreamCreateWithFlags(&m->compute_stream, cudaStreamNonBlocking));
    {
        int prio_lo = 0, prio_hi = 0;
        HN_CUDA_OK(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        HN_CUDA_OK(cudaStreamCreateWithPriority(&m->enc_stream, cudaStreamNonBlocking, prio_lo));
        // the recurrence's 16-CTA clusters must get their SMs as soon as a convolution kernel retires
        HN_CUDA_OK(cudaStreamCreateWithPriority(&m->rnn_stream, cudaStreamNonBlocking, prio_hi));
    }
    for (int i = 0; i < 2; ++i) {
        HN_CUDA_OK(cudaEventCreateWithFlags(&m->slot_ready[i], cudaEventDisableTiming));
        HN_CUDA_OK(cudaEventCreateWithFlags(&m->slot_done[i], cudaEventDisableTiming));
        HN_CUDA_OK(cudaEventCreateWithFlags(&m->async_done[i], cudaEventDisableTiming));
    }
    for (cudaEvent_t* e : {&m->ev_in, &m->ev_xfree, &m->ev_seq, &m->ev_rnn_last, &m->ev_plain_done})
        HN_CUDA_OK(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    *out = m.release();
    return 0;
}

int hn_model_num_tensors(const hn_model* m) { return m ? (int)m->slots.size() : 0; }

int hn_model_tensor_info(const hn_model* m, int i, const char** key, long long* numel) {
    HN_CHECK(m && i >= 0 && i < (int)m->slots.size(), "hn_model_tensor_info: bad index");
    if (key) *key = m->slots[i].key.c_str();
    if (numel) *numel = m->slots[i].numel;
    return 0;
}

int hn_model_set_tensor(hn_model* m, const char* key, const float* data, long long numel, int on_device) {
    HN_CHECK(m && key, "hn_model_set_tensor: NULL argument");
    auto it = m->index.find(key);
    if (it == m->index.end()) return fail(std::string("hn_model_set_tensor: unexpected key '") + key + "'");
    TensorSlot& s = m->slots[it->second];
    if (s.ignored) { s.set = true; return 0; }
    HN_CHECK(data != nullptr, "hn_model_set_tensor: data is NULL");
    if (numel != s.numel)
        return fail(std::string("hn_model_set_tensor: size mismatch for '") + key + "': got " + std::to_string(numel) +
                    ", expected " + std::to_string(s.numel));
    HN_ON_DEVICE(m->device);
    if (m->rnn_inflight) {        // forwards may still be running on the internal (non-blocking) streams: do not race them
        HN_CUDA_OK(cudaStreamSynchronize(m->enc_stream));
        HN_CUDA_OK(cudaStreamSynchronize(m->rnn_stream));
        m->rnn_inflight = false;
    }
    HN_CUDA_OK(cudaMemcpy(s.dev, data, (size_t)numel * sizeof(float),
                          on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice));
    s.set = true;
    m->finalized = false;
    return 0;
}

int hn_model_set_option(hn_model* m, const char* name, int value) {
    HN_CHECK(m && name, "hn_model_set_option: NULL argument");
    if (std::strcmp(name, "tensor_cores") == 0) { m->use_tc = value; return 0; }
    if (std::strcmp(name, "profile") == 0) { m->profile = value; return 0; }
    if (std::strcmp(name, "stem_tc") == 0) { m->stem_tc_on = value; return 0; }
    if (std::strcmp(name, "fuse_bottleneck") == 0) { m->fuse_on = value; return 0; }
    return fail(std::string("hn_model_set_option: unknown option '") + name + "'");
}

int hn_model_finalize(hn_model* m) {
    HN_CHECK(m, "hn_model_finalize: NULL model");
    for (auto& s : m->slots)
        if (!s.set && !s.ignored) return fail("hn_model_finalize: missing key '" + s.key + "' (strict load, utils.py:64)");
    HN_ON_DEVICE(m->device);
    cudaStream_t st = 0;
    if (pack_conv(m, m->stem, st)) return -1;
    if (!m->stem_wq && (m->alloc_t(&m->stem_wq, (size_t)2 * 64 * 224) || m->alloc_t(&m->stem_aux, 3 * 64 + 1))) return -1;
    if (stem_tc_pack_weights(m->T(m->stem.wkey), m->XP, m->stem_wq, m->stem.scale, m->stem.shift, m->stem_aux, st)) return -1;
    for (int l = 0; l < 4; ++l)
        for (auto& b : m->blocks[l]) {
            if (pack_conv(m, b.c1, st) || pack_conv(m, b.c2, st) || pack_conv(m, b.c3, st)) return -1;
            if (b.has_ds && pack_conv(m, b.ds, st)) return -1;
        }
    for (int s = 0; s < 4; ++s)
        for (int j = 0; j < 4; ++j)
            if (pack_conv(m, m->ghc[s][j], st)) return -1;
    for (int layer = 0; layer < 2; ++layer) {
        ConvLayer& c = m->xproj[layer];
        if (!c.w) {
            if (m->alloc_t(&c.w, (size_t)4096 * 1024) || m->alloc_t(&c.scale, 4096) || m->alloc_t(&c.shift, 4096)) return -1;
            if (m->alloc_t(&c.wq, (size_t)2 * 4096 * 1024) || m->alloc_t(&c.tc_scale, 3 * 4096 + 1)) return -1;
        }
        const std::string l = "_l" + std::to_string(layer);
        // [4096][1024] (fwd rows then reverse rows) -> [K=1024][N=4096]
        for (int dir = 0; dir < 2; ++dir) {
            const float* w = m->T("bi_rnn.weight_ih" + l + (dir ? "_reverse" : ""));
            HN_CUDA_OK(cudaMemcpyAsync(m->XP + (size_t)dir * 2048 * 1024, w, (size_t)2048 * 1024 * sizeof(float),
                                       cudaMemcpyDeviceToDevice, st));
            m->whh[layer][dir] = m->T("bi_rnn.weight_hh" + l + (dir ? "_reverse" : ""));
        }
        pack_oihw_kernel<<<(4096 * 1024 + 255) / 256, 256, 0, st>>>(m->XP, c.w, 4096, 1024, 1, 1);
        HN_LAUNCH_OK();

        lstm_bias_kernel<<<16, 256, 0, st>>>(m->T("bi_rnn.bias_ih" + l), m->T("bi_rnn.bias_hh" + l),
                                             m->T("bi_rnn.bias_ih" + l + "_reverse"),
                                             m->T("bi_rnn.bias_hh" + l + "_reverse"), c.scale, c.shift);
        HN_LAUNCH_OK();
        if (pack_weight_tc(m->XP, c.wq, c.scale, c.shift, c.tc_scale, c.tc_scale + 3 * 4096, 4096, 1024, 1, 1, st)) return -1;
        c.d.w = c.w; c.d.scale = c.scale; c.d.shift = c.shift;
    }
    HN_CUDA_OK(cudaMemcpyAsync(m->head_w, m->T("linear.weight"), 12 * 1024 * sizeof(float), cudaMemcpyDeviceToDevice, st));
    HN_CUDA_OK(cudaMemcpyAsync(m->head_b, m->T("linear.bias"), 12 * sizeof(float), cudaMemcpyDeviceToDevice, st));
    HN_CUDA_OK(cudaStreamSynchronize(st));
    m->bn_stale = false;
    m->finalized = true;
    return 0;
}

// ---- the three parts of HorizonNet.forward (model.py:254-281); static helpers (no extern "C" linkage needed)
// (1) normalise + stem + max-pool + layer1..4 + the 16 height-reduction convs: leaves gout[] in GO[0..3]
static int forward_encoder(hn_model* m, const float* x, int B, int in_channels, Act gout[4], cudaStream_t st,
                           cudaEvent_t x_consumed, const TrainCtx* tr = nullptr) {
    if (m->bn_stale) {
        bool need = !tr;                     // eval forward, or a train forward with frozen (eval-mode) BN modules
        for (size_t i = 0; tr && i < m->bn_names.size(); ++i) need = need || !tr->bn_train[i];
        if (need && refold_bn(m, st)) return -1;
    }
    // model.py:248-252 + :73-76: normalise, stem conv/BN/ReLU, max-pool
    Act s0 = mk(m->S0, B, 256, 512, 64);
    {
        Scope sc(m, CLS_STEM, 2.0 * B * 256 * 512 * 64 * 147, st);
        const bool tc = m->use_tc && m->stem_tc_on;
        const bool batch_stats = tr && tr->bn_train[m->stem.bn_index];
        const float *scale = m->stem.scale, *shift = m->stem.shift, *aux = m->stem_aux;
        for (int pass = batch_stats ? 0 : 1; pass < 2; ++pass) {
            if (batch_stats) {          // pass 0: raw stem output -> batch statistics; pass 1: the real thing
                if (pass == 0 && bn_identity_constants(nullptr, m->trn_scale, m->trn_shift, 64, st)) return -1;
                if (pass == 1) {
                    if (bn_batch_stats(s0, false, m->trn_sums, st)) return -1;
                    if (bn_train_finalize(m->trn_sums, (long long)B * 256 * 512, m->T(m->stem.bnprefix + ".weight"),
                                          m->T(m->stem.bnprefix + ".bias"), nullptr,
                                          const_cast<float*>(m->T(m->stem.bnprefix + ".running_mean")),
                                          const_cast<float*>(m->T(m->stem.bnprefix + ".running_var")),
                                          tr->bn_factor[m->stem.bn_index], m->trn_scale, m->trn_shift, 64, st))
                        return -1;
                }
                if (tc && tc_aux_update(m->trn_scale, m->trn_shift, m->stem_aux + 3 * 64, m->trn_aux, 64, st)) return -1;
                scale = m->trn_scale; shift = m->trn_shift; aux = m->trn_aux;
            }
            if (tc) {
                // packed input planes live in X[0] (free until layer1): B * 8.6 MB of its B * 33.8 MB
                if (stem_tc(x, B, in_channels, m->stem_wq, aux, shift, reinterpret_cast<unsigned short*>(m->X[0]), s0, st,
                            pass == 1)) return -1;
            } else if (stem_f32(x, B, in_channels, m->stem.w, scale, shift, s0, st, pass == 1)) return -1;
        }
    }
    if (x_consumed) HN_CUDA_OK(cudaEventRecord(x_consumed, st));       // the input batch is not read after the stem
    Act cur = mk(m->S1, B, 128, 256, 64);
    {
        Scope sc(m, CLS_POOL, 0.0, st);
        if (maxpool3x3s2(s0, cur, st, m->use_tc != 0)) return -1;
    }

    // model.py:78-81: layer1..layer4 (torchvision Bottleneck v1.5)
    Act feats[4];
    for (int l = 0; l < 4; ++l) {
        const int nb = (int)m->blocks[l].size();
        for (int b = 0; b < nb; ++b) {
            const hn_model::Block& blk = m->blocks[l][b];
            const int s = blk.c2.d.sh;
            const int Ho = cur.H / s, Wo = cur.W / s;
            Act t1 = mk(m->T1, B, cur.H, cur.W, blk.c1.d.Cout);
            Act t2 = mk(m->T2, B, Ho, Wo, blk.c2.d.Cout);
            Act y = mk(b == nb - 1 ? m->F[l] : m->X[b & 1], B, Ho, Wo, blk.c3.d.Cout);
            if (conv_bn(m, blk.c1, cur, t1, nullptr, st, CLS_ENC_CONV, tr)) return -1;
            const float* idn = cur.p;
            if (blk.has_ds) {
                Act d = mk(m->IDN, B, Ho, Wo, blk.ds.d.Cout);
                if (conv_bn(m, blk.ds, cur, d, nullptr, st, CLS_ENC_CONV, tr)) return -1;
                idn = d.p;
            }
            if (!tr && m->use_tc && m->fuse_on && blk.c2.wq && blk.c3.wq && bott_tc_supported(blk.c2.d, blk.c3.d, t1, y)) {
                // layer1: conv2 + conv3 in one kernel, the 64-channel intermediate stays in shared memory (conv_tc.cu)
                const double flops = 2.0 * (double)B * Ho * Wo * (64.0 * 9 * 64 + (double)blk.c3.d.Cout * 64);
                Scope sc(m, CLS_ENC_CONV, flops, st);
                if (bott_tc_planes(blk.c2.d, blk.c2.wq, blk.c2.tc_scale, blk.c3.d, blk.c3.wq, blk.c3.tc_scale, t1,
                                   reinterpret_cast<const unsigned short*>(t1.p), y, reinterpret_cast<unsigned short*>(y.p),
                                   reinterpret_cast<const unsigned short*>(idn), st))
                    return -1;
            } else {
                if (conv_bn(m, blk.c2, t1, t2, nullptr, st, CLS_ENC_CONV, tr)) return -1;
                if (conv_bn(m, blk.c3, t2, y, idn, st, CLS_ENC_CONV, tr)) return -1;   // + identity, ReLU
            }
            cur = y;
        }
        feats[l] = cur;
    }

    // model.py:148-151: 4 x (3x3 stride (2,1) conv + bias + BN + ReLU) per scale
    for (int s = 0; s < 4; ++s) {
        Act g = feats[s];
        for (int j = 0; j < 4; ++j) {
            const ConvLayer& c = m->ghc[s][j];
            Act o = mk(j == 3 ? m->GO[s] : m->G[j & 1], B, g.H / 2, g.W, c.d.Cout);
            if (conv_bn(m, c, g, o, nullptr, st, CLS_GHC_CONV, tr)) return -1;
            g = o;
        }
        gout[s] = g;
    }
    return 0;
}

// (2) model.py:152-155 + :175-178 + :263: upsample + flatten + concat + permute -> SEQ [T=256][B][1024]
static int forward_sequence(hn_model* m, const Act gout[4], cudaStream_t st) {
    Scope sc(m, CLS_TAIL, 0.0, st);
    return ghc_to_sequence(gout, m->SEQ, st, m->use_tc != 0);
}

// (3) model.py:264-281: 2-layer bidirectional LSTM (eval: dropout = identity), linear head, reshape, split
static int forward_rnn(hn_model* m, int B, float* bon, float* cor, cudaStream_t st, const TrainCtx* tr = nullptr) {
    const float* lin = m->SEQ;
    float* louts[2] = {m->R1, m->R2};
    for (int layer = 0; layer < 2; ++layer) {
        Act a = mk(const_cast<float*>(lin), 1, 1, 256 * B, 1024, 0);
        Act xp = mk(m->XP, 1, 1, 256 * B, 4096, 0);
        if (tr && layer == 1 && tr->rnn_p > 0.0) {
            // train mode: nn.LSTM(dropout=p) zeroes layer-1 outputs on their way into layer 2 (model.py:226)
            Scope sc(m, CLS_TAIL, 0.0, st);
            if (tr->mask[0] ? multiply_inplace(m->R1, tr->mask[0], (size_t)256 * B * 1024, st)
                            : dropout_inplace(m->R1, (size_t)256 * B * 1024, tr->rnn_p, tr->seed, 0, false, st))
                return -1;
        }
        if (m->use_tc && layer == 1) {
            // layer-2 projection operand: the fp32 recurrence output as fp16 hi/lo planes
            Scope sc(m, CLS_TAIL, 0.0, st);
            if (split_planes(m->R1, reinterpret_cast<unsigned short*>(m->R1S), (size_t)256 * B * 1024, st)) return -1;
            a.p = m->R1S;
        }
        if (run_conv(m, m->xproj[layer], a, xp, nullptr, st, CLS_XPROJ, true)) return -1;
        {
            Scope sc(m, CLS_LSTM, 2.0 * 256 * B * 2 * 2048 * 512, st);
            if (lstm_layer(m->XP, m->whh[layer][0], m->whh[layer][1], louts[layer], 256, B, m->counters,
                           m->error_flag, st))
                return -1;
        }
        lin = louts[layer];
    }
    if (tr && tr->head_p > 0.0) {         // train mode: self.drop_out before the linear head (model.py:265)
        Scope sc(m, CLS_TAIL, 0.0, st);
        if (tr->mask[1] ? multiply_inplace(m->R2, tr->mask[1], (size_t)256 * B * 1024, st)
                        : dropout_inplace(m->R2, (size_t)256 * B * 1024, tr->head_p, tr->seed, 1, false, st))
            return -1;
    }
    {
        Scope sc(m, CLS_HEAD, 2.0 * 256 * B * 12 * 1024, st);
        if (linear_head(m->R2, m->head_w, m->head_b, bon, cor, 256, B, st)) return -1;
    }
    return 0;
}

static int forward_args_ok(hn_model* m, const void* x, int B, const void* bon, const void* cor, const char* who) {
    if (!(m && x && bon && cor)) return fail(std::string(who) + ": NULL argument");
    if (!m->finalized) return fail(std::string(who) + ": call hn_model_finalize after setting all tensors");
    if (!(B >= 1 && B <= m->max_batch)) return fail(std::string(who) + ": batch exceeds max_batch given at create");
    return 0;
}

// Two-stream enqueue of one forward: encoder + height reduction on enc_stream (the caller has already made
// enc_stream wait for the input), sequence assembly once the previous batch's recurrence no longer reads SEQ,
// then projections + recurrence + head on rnn_stream.  `done` (optional) is recorded when bon/cor are complete.
static int enqueue_two_stream(hn_model* m, const float* x, int B, int in_channels, float* bon, float* cor,
                              cudaEvent_t done) {
    if (m->plain_recorded) {      // a plain hn_model_forward on a caller stream may still use the workspace
        HN_CUDA_OK(cudaStreamWaitEvent(m->enc_stream, m->ev_plain_done, 0));
        HN_CUDA_OK(cudaStreamWaitEvent(m->rnn_stream, m->ev_plain_done, 0));
        m->plain_recorded = false;
    }
    Act gout[4];
    if (forward_encoder(m, x, B, in_channels, gout, m->enc_stream, m->ev_xfree)) return -1;
    if (m->rnn_inflight) HN_CUDA_OK(cudaStreamWaitEvent(m->enc_stream, m->ev_rnn_last, 0));
    if (forward_sequence(m, gout, m->enc_stream)) return -1;
    HN_CUDA_OK(cudaEventRecord(m->ev_seq, m->enc_stream));
    HN_CUDA_OK(cudaStreamWaitEvent(m->rnn_stream, m->ev_seq, 0));
    if (forward_rnn(m, B, bon, cor, m->rnn_stream)) return -1;
    HN_CUDA_OK(cudaEventRecord(m->ev_rnn_last, m->rnn_stream));
    if (done) HN_CUDA_OK(cudaEventRecord(done, m->rnn_stream));
    m->rnn_inflight = true;
    m->last_batch = B;
    return 0;
}

int hn_model_forward(hn_model* m, const float* x, int B, int in_channels, float* bon, float* cor, void* stream) {
    if (forward_args_ok(m, x, B, bon, cor, "hn_model_forward")) return -1;
    HN_ON_DEVICE(m->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (m->rnn_inflight) {        // join batches still in flight on the internal streams (they share the workspace)
        HN_CUDA_OK(cudaStreamWaitEvent(st, m->ev_rnn_last, 0));
        m->rnn_inflight = false;
    }
    m->last_batch = B;
    Act gout[4];
    if (forward_encoder(m, x, B, in_channels, gout, st, nullptr)) return -1;
    if (forward_sequence(m, gout, st)) return -1;
    if (forward_rnn(m, B, bon, cor, st)) return -1;
    HN_CUDA_OK(cudaEventRecord(m->ev_plain_done, st));
    m->plain_recorded = true;
    return 0;
}

int hn_model_num_bn(const hn_model* m) { return m ? (int)m->bn_names.size() : 0; }

const char* hn_model_bn_name(const hn_model* m, int i) {
    return (m && i >= 0 && i < (int)m->bn_names.size()) ? m->bn_names[i].c_str() : nullptr;
}

int hn_model_forward_train(hn_model* m, const float* x, int B, int in_channels, float* bon, float* cor,
                           const unsigned char* bn_train, const double* bn_factor, int n_bn, unsigned long long seed,
                           double rnn_dropout, double head_dropout, const float* rnn_mask, const float* head_mask,
                           void* stream) {
    if (forward_args_ok(m, x, B, bon, cor, "hn_model_forward_train")) return -1;
    HN_CHECK(bn_train && bn_factor && n_bn == (int)m->bn_names.size(),
             "hn_model_forward_train: bn_train / bn_factor need hn_model_num_bn() entries");
    HN_CHECK(rnn_dropout >= 0.0 && rnn_dropout < 1.0 && head_dropout >= 0.0 && head_dropout < 1.0,
             "hn_model_forward_train: dropout probabilities must be in [0, 1)");
    HN_ON_DEVICE(m->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (m->rnn_inflight) {
        HN_CUDA_OK(cudaStreamWaitEvent(st, m->ev_rnn_last, 0));
        m->rnn_inflight = false;
    }
    m->last_batch = B;
    const TrainCtx tr{bn_train, bn_factor, seed, rnn_dropout, head_dropout, {rnn_mask, head_mask}};
    Act gout[4];
    if (forward_encoder(m, x, B, in_channels, gout, st, nullptr, &tr)) return -1;
    if (forward_sequence(m, gout, st)) return -1;
    if (forward_rnn(m, B, bon, cor, st, &tr)) return -1;
    for (int i = 0; i < n_bn; ++i) m->bn_stale = m->bn_stale || (bn_train[i] && bn_factor[i] >= 0.0);
    HN_CUDA_OK(cudaEventRecord(m->ev_plain_done, st));
    m->plain_recorded = true;
    return 0;
}

int hn_model_get_tensor(hn_model* m, const char* key, float* out, long long numel, int on_device, void* stream) {
    HN_CHECK(m && key && out, "hn_model_get_tensor: NULL argument");
    auto it = m->index.find(key);
    if (it == m->index.end()) return fail(std::string("hn_model_get_tensor: unknown key '") + key + "'");
    const TensorSlot& s = m->slots[it->second];
    HN_CHECK(!s.ignored && s.set && s.dev, "hn_model_get_tensor: tensor was never set");
    HN_CHECK(numel == s.numel, "hn_model_get_tensor: element count differs from the tensor's");
    HN_ON_DEVICE(m->device);
    cudaStream_t st = (cudaStream_t)stream;
    HN_CUDA_OK(cudaMemcpyAsync(out, s.dev, (size_t)numel * sizeof(float),
                               on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
    if (!on_device) HN_CUDA_OK(cudaStreamSynchronize(st));
    return 0;
}

int hn_dropout_mask(unsigned long long seed, int which, double p, float* out, long long n, void* stream) {
    HN_CHECK(out && n >= 0, "hn_dropout_mask: bad argument");
    return dropout_inplace(out, (size_t)n, p, seed, which, true, (cudaStream_t)stream);
}

int hn_model_forward_async(hn_model* m, const float* x, int B, int in_channels, float* bon, float* cor, void* stream) {
    if (forward_args_ok(m, x, B, bon, cor, "hn_model_forward_async")) return -1;
    HN_ON_DEVICE(m->device);
    cudaStream_t st = (cudaStream_t)stream;
    HN_CUDA_OK(cudaEventRecord(m->ev_in, st));                          // x (and everything before it on st) is ready
    HN_CUDA_OK(cudaStreamWaitEvent(m->enc_stream, m->ev_in, 0));
    const int slot = (int)(m->async_count & 1);
    const bool had_prev = m->async_count > 0;
    if (enqueue_two_stream(m, x, B, in_channels, bon, cor, m->async_done[slot])) return -1;
    HN_CUDA_OK(cudaStreamWaitEvent(st, m->ev_xfree, 0));                // x may be overwritten by later work on st
    if (had_prev) HN_CUDA_OK(cudaStreamWaitEvent(st, m->async_done[slot ^ 1], 0));   // outputs of the PREVIOUS call
    ++m->async_count;
    return 0;
}

int hn_model_flush(hn_model* m, void* stream) {
    HN_CHECK(m, "hn_model_flush: NULL model");
    HN_ON_DEVICE(m->device);
    if (m->rnn_inflight) HN_CUDA_OK(cudaStreamWaitEvent((cudaStream_t)stream, m->ev_rnn_last, 0));
    return 0;
}

int hn_model_profile_read(hn_model* m, double* ms, double* flops, long long* launches, int reset) {
    HN_CHECK(m, "hn_model_profile_read: NULL model");
    HN_ON_DEVICE(m->device);
    for (auto& sp : m->spans) {
        HN_CUDA_OK(cudaEventSynchronize(sp.b));
        float t = 0.f;
        HN_CUDA_OK(cudaEventElapsedTime(&t, sp.a, sp.b));
        m->prof_ms[sp.cls] += t; m->prof_flops[sp.cls] += sp.flops; m->prof_launches[sp.cls] += 1;
        m->free_events.push_back(sp.a); m->free_events.push_back(sp.b);
    }
    m->spans.clear();
    for (int i = 0; i < HN_NUM_CLASSES; ++i) {
        if (ms) ms[i] = m->prof_ms[i];
        if (flops) flops[i] = m->prof_flops[i];
        if (launches) launches[i] = m->prof_launches[i];
        if (reset) { m->prof_ms[i] = 0; m->prof_flops[i] = 0; m->prof_launches[i] = 0; }
    }
    return 0;
}

int hn_model_check(hn_model* m) {
    // surfaces device-side failures (LSTM spin timeout) after a synchronisation point
    HN_CHECK(m, "hn_model_check: NULL model");
    HN_ON_DEVICE(m->device);
    int flag = 0;
    HN_CUDA_OK(cudaMemcpy(&flag, m->error_flag, sizeof(int), cudaMemcpyDeviceToHost));
    if (flag) {
        cudaMemset(m->error_flag, 0, sizeof(int));
        return fail("hn_model: the persistent LSTM kernel timed out waiting for a peer CTA");
    }
    return 0;
}

int hn_model_forward_host(hn_model* m, const float* x, int B, int in_channels, float* bon, float* cor) {
    HN_CHECK(m && x && bon && cor, "hn_model_forward_host: NULL argument");
    HN_CHECK(B >= 1 && B <= m->max_batch, "hn_model_forward_host: batch exceeds max_batch");
    HN_CHECK(in_channels >= 3, "hn_model_forward_host: need >= 3 channels");
    HN_CHECK(m->submit_count == m->collect_count, "hn_model_forward_host: collect the submitted batches first");
    HN_ON_DEVICE(m->device);
    cudaStream_t st = 0;
    // only the first 3 channels are used (model.py:252): copy them image by image
    for (int b = 0; b < B; ++b)
        HN_CUDA_OK(cudaMemcpyAsync(m->x_in + (size_t)b * 3 * 512 * 1024, x + (size_t)b * in_channels * 512 * 1024,
                                   (size_t)3 * 512 * 1024 * sizeof(float), cudaMemcpyHostToDevice, st));
    if (hn_model_forward(m, m->x_in, B, 3, m->bon_out, m->cor_out, st)) return -1;
    HN_CUDA_OK(cudaMemcpyAsync(bon, m->bon_out, (size_t)B * 2 * 1024 * sizeof(float), cudaMemcpyDeviceToHost, st));
    HN_CUDA_OK(cudaMemcpyAsync(cor, m->cor_out, (size_t)B * 1024 * sizeof(float), cudaMemcpyDeviceToHost, st));
    HN_CUDA_OK(cudaStreamSynchronize(st));
    return hn_model_check(m);
}

int hn_model_submit_host(hn_model* m, const float* x, int B, int in_channels) {
    HN_CHECK(m && x, "hn_model_submit_host: NULL argument");
    HN_CHECK(m->finalized, "hn_model_submit_host: call hn_model_finalize after setting all tensors");
    HN_CHECK(B >= 1 && B <= m->max_batch, "hn_model_submit_host: batch exceeds max_batch");
    HN_CHECK(in_channels >= 3, "hn_model_submit_host: need >= 3 channels");
    HN_CHECK(m->submit_count - m->collect_count < 2, "hn_model_submit_host: both input slots are in flight (collect first)");
    HN_ON_DEVICE(m->device);
    const int slot = m->submit_count & 1;
    // the slot's previous batch was collected (fully synchronised), so its input buffer is free
    for (int b = 0; b < B; ++b)
        HN_CUDA_OK(cudaMemcpyAsync(m->x_slot[slot] + (size_t)b * 3 * 512 * 1024, x + (size_t)b * in_channels * 512 * 1024,
                                   (size_t)3 * 512 * 1024 * sizeof(float), cudaMemcpyHostToDevice, m->copy_stream));
    HN_CUDA_OK(cudaEventRecord(m->slot_ready[slot], m->copy_stream));
    // the forward is enqueued right away: the encoder of this batch overlaps the recurrence of the previous one
    HN_CUDA_OK(cudaStreamWaitEvent(m->enc_stream, m->slot_ready[slot], 0));
    if (enqueue_two_stream(m, m->x_slot[slot], B, 3, m->bon_slot[slot], m->cor_slot[slot], m->slot_done[slot])) return -1;
    m->slot_batch[slot] = B;
    ++m->submit_count;
    return 0;
}

int hn_model_collect_host(hn_model* m, float* bon, float* cor) {
    HN_CHECK(m && bon && cor, "hn_model_collect_host: NULL argument");
    HN_CHECK(m->collect_count < m->submit_count, "hn_model_collect_host: nothing submitted");
    HN_ON_DEVICE(m->device);
    const int slot = m->collect_count & 1;
    const int B = m->slot_batch[slot];
    cudaStream_t st = m->compute_stream;
    HN_CUDA_OK(cudaStreamWaitEvent(st, m->slot_done[slot], 0));
    HN_CUDA_OK(cudaMemcpyAsync(bon, m->bon_slot[slot], (size_t)B * 2 * 1024 * sizeof(float), cudaMemcpyDeviceToHost, st));
    HN_CUDA_OK(cudaMemcpyAsync(cor, m->cor_slot[slot], (size_t)B * 1024 * sizeof(float), cudaMemcpyDeviceToHost, st));
    // a device-side LSTM timeout of this batch is surfaced here (the flag is written before the outputs complete)
    int flag = 0;
    HN_CUDA_OK(cudaMemcpyAsync(&flag, m->error_flag, sizeof(int), cudaMemcpyDeviceToHost, st));
    HN_CUDA_OK(cudaStreamSynchronize(st));
    ++m->collect_count;
    if (flag) {
        cudaMemsetAsync(m->error_flag, 0, sizeof(int), st);
        cudaStreamSynchronize(st);
        return fail("hn_model: the persistent LSTM kernel timed out waiting for a peer CTA");
    }
    return 0;
}

int hn_model_infer_tta(hn_model* m, const float* x, int in_channels, int flip, const int* shifts, int n_rotate,
                       float* y_bon_pix, float* y_cor, void* stream) {
    HN_CHECK(m && x && y_bon_pix && y_cor, "hn_model_infer_tta: NULL argument");
    HN_CHECK(in_channels == 3, "hn_model_infer_tta: expects a 3-channel panorama (inference.py:196-200)");
    HN_CHECK(n_rotate >= 0 && n_rotate <= 32 && (n_rotate == 0 || shifts), "hn_model_infer_tta: bad rotate list");
    const int V = 1 + (flip ? 1 : 0) + n_rotate;
    HN_CHECK(V <= m->max_batch && V <= 64, "hn_model_infer_tta: views exceed max_batch");
    HN_CHECK(m->submit_count == m->collect_count, "hn_model_infer_tta: collect the submitted batches first");
    HN_ON_DEVICE(m->device);
    cudaStream_t st = (cudaStream_t)stream;
    int host[128];
    int v = 0;
    host[v] = 0; host[64 + v] = 0; ++v;                         // aug_type '' (inference.py:34)
    if (flip) { host[v] = 1; host[64 + v] = 0; ++v; }           // 'flip' (:36-38)
    for (int i = 0; i < n_rotate; ++i, ++v) { host[v] = 2; host[64 + v] = shifts[i]; }   // 'rotate shift' (:39-42)
    HN_CUDA_OK(cudaMemcpyAsync(m->tta_ints, host, sizeof(host), cudaMemcpyHostToDevice, st));
    HN_CUDA_OK(cudaStreamSynchronize(st));                      // host[] is a stack array
    if (tta_views(x, m->x_slot[1], 1, V, m->tta_ints, m->tta_ints + 64, st)) return -1;
    if (hn_model_forward(m, m->x_slot[1], V, 3, m->bon_out, m->cor_out, st)) return -1;
    return tta_merge(m->bon_out, m->cor_out, 1, V, m->tta_ints, m->tta_ints + 64, y_bon_pix, y_cor, st);
}

long long hn_layout_workspace_bytes(int B) { return B >= 1 ? (long long)hn::layout_workspace_bytes(B) : 0; }

int hn_layout(const float* y_bon_pix, const float* y_cor, int B, int mode, float min_v, int r_px, void* workspace,
              float* cor_id, int* n_cor, float* z1, int* status, int* peaks, int* types, void* stream) {
    HN_CHECK(y_bon_pix && y_cor && workspace && cor_id && n_cor && z1 && status, "hn_layout: NULL argument");
    HN_CHECK(B >= 1 && B <= 65535, "hn_layout: batch must be in 1..65535");
    HN_CHECK(mode >= HN_LAYOUT_GENERAL && mode <= HN_LAYOUT_RAW, "hn_layout: mode must be general, cuboid or raw");
    HN_CHECK(mode == HN_LAYOUT_RAW || r_px >= 1, "hn_layout: the peak window r_px must be >= 1");
    return layout(y_bon_pix, y_cor, B, mode, min_v, r_px, workspace, cor_id, n_cor, z1, status, peaks, types,
                  (cudaStream_t)stream);
}

int hn_model_infer_layout(hn_model* m, const float* x, int B, int flip, const int* shifts, int n_rotate, int mode,
                          float min_v, int r_px, void* workspace, float* y_bon_pix, float* y_cor, float* cor_id,
                          int* n_cor, float* z1, int* status, int* peaks, int* types, void* stream) {
    HN_CHECK(m && x && y_bon_pix && y_cor, "hn_model_infer_layout: NULL argument");
    HN_CHECK(B >= 1, "hn_model_infer_layout: batch must be >= 1");
    HN_CHECK(n_rotate >= 0 && n_rotate <= 32 && (n_rotate == 0 || shifts), "hn_model_infer_layout: bad rotate list");
    const int V = 1 + (flip ? 1 : 0) + n_rotate;
    HN_CHECK(V <= m->max_batch, "hn_model_infer_layout: views exceed max_batch");
    HN_CHECK(m->submit_count == m->collect_count, "hn_model_infer_layout: collect the submitted batches first");
    HN_ON_DEVICE(m->device);
    cudaStream_t st = (cudaStream_t)stream;
    int host[128];
    int v = 0;
    host[v] = 0; host[64 + v] = 0; ++v;                         // same view list as hn_model_infer_tta
    if (flip) { host[v] = 1; host[64 + v] = 0; ++v; }
    for (int i = 0; i < n_rotate; ++i, ++v) { host[v] = 2; host[64 + v] = shifts[i]; }
    HN_CUDA_OK(cudaMemcpyAsync(m->tta_ints, host, sizeof(host), cudaMemcpyHostToDevice, st));
    HN_CUDA_OK(cudaStreamSynchronize(st));                      // host[] is a stack array
    const int chunk = m->max_batch / V;                         // chunk * V views per forward
    const size_t per = (size_t)3 * 512 * 1024;
    for (int b0 = 0; b0 < B; b0 += chunk) {
        const int nb = B - b0 < chunk ? B - b0 : chunk;
        const float* xin = x + b0 * per;
        if (V > 1) {
            if (tta_views(xin, m->x_slot[1], nb, V, m->tta_ints, m->tta_ints + 64, st)) return -1;
            xin = m->x_slot[1];
        }
        if (hn_model_forward(m, xin, nb * V, 3, m->bon_out, m->cor_out, st)) return -1;
        if (tta_merge(m->bon_out, m->cor_out, nb, V, m->tta_ints, m->tta_ints + 64, y_bon_pix + (size_t)b0 * 2 * 1024,
                      y_cor + (size_t)b0 * 1024, st))
            return -1;
    }
    return hn_layout(y_bon_pix, y_cor, B, mode, min_v, r_px, workspace, cor_id, n_cor, z1, status, peaks, types, stream);
}

int hn_model_stage(hn_model* m, const char* stage, float* out, long long capacity, int dims[4], void* stream) {
    HN_CHECK(m && stage && out && dims, "hn_model_stage: NULL argument");
    HN_CHECK(m->last_batch > 0, "hn_model_stage: no forward has run yet");
    HN_ON_DEVICE(m->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (m->rnn_inflight) HN_CUDA_OK(cudaStreamWaitEvent(st, m->ev_rnn_last, 0));
    const int B = m->last_batch;
    const std::string s(stage);
    for (int l = 0; l < 4; ++l)
        if (s == "layer" + std::to_string(l + 1)) {
            const int C = 256 << l, H = 128 >> l, W = 256 >> l;
            const size_t total = (size_t)B * C * H * W;
            HN_CHECK((long long)total <= capacity, "hn_model_stage: output buffer too small");
            const float* src = m->F[l];
            if (m->use_tc) {       // F[l] holds fp16 hi/lo planes: merge into X[0] (free after the forward)
                const size_t n = (size_t)B * H * (W + 2) * C;
                float* tmp = m->X[0];
                HN_CHECK(n <= (size_t)m->max_batch * 128 * 258 * 256, "hn_model_stage: scratch buffer too small");
                if (merge_planes(reinterpret_cast<const unsigned short*>(m->F[l]), tmp, n, st)) return -1;
                src = tmp;
            }
            nhwc_to_nchw_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(src, out, B, H, W, C, 1);
            HN_LAUNCH_OK();
            dims[0] = B; dims[1] = C; dims[2] = H; dims[3] = W;
            return 0;
        }
    if (s == "stem") {           // conv1 + bn1 + relu (model.py:73-75), before the max-pool; S0 is fp32 on both paths
        const size_t n = (size_t)B * 64 * 256 * 512;
        HN_CHECK((long long)n <= capacity, "hn_model_stage: output buffer too small");
        nhwc_to_nchw_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(m->S0, out, B, 256, 512, 64, 1);
        HN_LAUNCH_OK();
        dims[0] = B; dims[1] = 64; dims[2] = 256; dims[3] = 512;
        return 0;
    }
    const size_t total = (size_t)256 * B * 1024;
    HN_CHECK((long long)total <= capacity, "hn_model_stage: output buffer too small");
    if (s == "feature") {
        const float* seq = m->SEQ;
        if (m->use_tc) {      // SEQ holds fp16 hi/lo planes; XP is dead after the forward and large enough
            if (merge_planes(reinterpret_cast<const unsigned short*>(m->SEQ), m->XP, total, st)) return -1;
            seq = m->XP;
        }
        seq_to_feature_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(seq, out, 256, B);
        HN_LAUNCH_OK();
        dims[0] = B; dims[1] = 1024; dims[2] = 256; dims[3] = 0;
        return 0;
    }
    if (s == "rnn_out") {
        HN_CUDA_OK(cudaMemcpyAsync(out, m->R2, total * sizeof(float), cudaMemcpyDeviceToDevice, st));
        dims[0] = 256; dims[1] = B; dims[2] = 1024; dims[3] = 0;
        return 0;
    }
    return fail("hn_model_stage: unknown stage '" + s + "'");
}

void hn_model_destroy(hn_model* m) { delete m; }

// ---- pano_stretch ------------------------------------------------------------------------------
static int pano_stretch_any(const void* img, void* out, int f64, int n, int h, int w, int c, const double* kx, const double* ky,
                            int order, void* stream, const char* who) {
    if (!(n >= 0 && h >= 1 && w >= 1)) return fail(std::string(who) + ": bad geometry");
    if (n == 0) return 0;
    if (!(img && out && kx && ky)) return fail(std::string(who) + ": NULL argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(std::string(who) + ": no CUDA device -- libhorizonnet_b200 has no CPU path");
    for (int i = 0; i < n; ++i)
        if (!(kx[i] > 0 && ky[i] > 0)) return fail(std::string(who) + ": kx, ky must be positive");
    cudaStream_t st = (cudaStream_t)stream;
    double* scratch = nullptr;
    const size_t nd = (size_t)2 * n + (size_t)4 * n * w + h;
    HN_CUDA_OK(cudaMallocAsync(reinterpret_cast<void**>(&scratch), nd * sizeof(double), st));
    HN_CUDA_OK(cudaMemcpyAsync(scratch, kx, n * sizeof(double), cudaMemcpyHostToDevice, st));
    HN_CUDA_OK(cudaMemcpyAsync(scratch + n, ky, n * sizeof(double), cudaMemcpyHostToDevice, st));
    int rc = f64 ? pano_stretch_device_f64(static_cast<const double*>(img), static_cast<double*>(out), n, h, w, c, scratch,
                                           scratch + n, scratch + 2 * (size_t)n, order, st)
                 : pano_stretch_device(static_cast<const float*>(img), static_cast<float*>(out), n, h, w, c, scratch,
                                       scratch + n, scratch + 2 * (size_t)n, order, st);
    cudaFreeAsync(scratch, st);
    return rc;
}

static int pano_stretch_any_host(const void* img, void* out, int f64, int n, int h, int w, int c, const double* kx,
                                 const double* ky, int order, const char* who) {
    if (n == 0) return 0;
    if (!(img && out && kx && ky)) return fail(std::string(who) + ": NULL argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(std::string(who) + ": no CUDA device -- libhorizonnet_b200 has no CPU path");
    const size_t bytes = (size_t)n * h * w * c * (f64 ? sizeof(double) : sizeof(float));
    void *d_in = nullptr, *d_out = nullptr;
    HN_CUDA_OK(cudaMalloc(&d_in, bytes));
    if (cudaMalloc(&d_out, bytes) != cudaSuccess) { cudaFree(d_in); return fail(std::string(who) + ": out of memory"); }
    int rc = 0;
    if (cudaMemcpy(d_in, img, bytes, cudaMemcpyHostToDevice) != cudaSuccess) rc = fail(std::string(who) + ": H2D failed");
    if (!rc) rc = pano_stretch_any(d_in, d_out, f64, n, h, w, c, kx, ky, order, nullptr, who);
    if (!rc && cudaMemcpy(out, d_out, bytes, cudaMemcpyDeviceToHost) != cudaSuccess) rc = fail(std::string(who) + ": D2H failed");
    cudaFree(d_in);
    cudaFree(d_out);
    return rc;
}

int hn_pano_stretch(const float* img, float* out, int n, int h, int w, int c, const double* kx, const double* ky,
                    int order, void* stream) {
    return pano_stretch_any(img, out, 0, n, h, w, c, kx, ky, order, stream, "hn_pano_stretch");
}
int hn_pano_stretch_host(const float* img, float* out, int n, int h, int w, int c, const double* kx,
                         const double* ky, int order) {
    return pano_stretch_any_host(img, out, 0, n, h, w, c, kx, ky, order, "hn_pano_stretch_host");
}
int hn_pano_stretch_f64(const double* img, double* out, int n, int h, int w, int c, const double* kx, const double* ky,
                        int order, void* stream) {
    return pano_stretch_any(img, out, 1, n, h, w, c, kx, ky, order, stream, "hn_pano_stretch_f64");
}
int hn_pano_stretch_host_f64(const double* img, double* out, int n, int h, int w, int c, const double* kx,
                             const double* ky, int order) {
    return pano_stretch_any_host(img, out, 1, n, h, w, c, kx, ky, order, "hn_pano_stretch_host_f64");
}

// ---- training augmentation, image path (reference dataset.py:53, 69-105, 124) ----------------------
int hn_augment(const unsigned char* img, float* out, int n, int h, int w, const double* kx, const double* ky,
               const int* flip, const int* dx, const float* gamma, void* stream) {
    HN_CHECK(n >= 0 && h >= 1 && w >= 1, "hn_augment: bad geometry");
    if (n == 0) return 0;
    HN_CHECK(img && out, "hn_augment: NULL argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail("hn_augment: no CUDA device -- libhorizonnet_b200 has no CPU path");
    std::vector<double> k((size_t)2 * n, 1.0);
    std::vector<int> prm((size_t)4 * n, 0);
    for (int i = 0; i < n; ++i) {
        const bool stretch = kx && ky && kx[i] > 0 && ky[i] > 0;
        if (kx && ky) HN_CHECK((kx[i] > 0) == (ky[i] > 0), "hn_augment: kx and ky must both be positive, or both <= 0 (no stretch)");
        if (stretch) { k[i] = kx[i]; k[(size_t)n + i] = ky[i]; }
        const int d = dx ? dx[i] : 0;
        HN_CHECK(d >= 0 && d < w, "hn_augment: dx must be in [0, W) (dataset.py:95 np.random.randint(W))");
        const float g = gamma ? gamma[i] : 0.f;
        prm[(size_t)4 * i + 0] = (flip && flip[i]) ? 1 : 0;
        prm[(size_t)4 * i + 1] = d;
        std::memcpy(&prm[(size_t)4 * i + 2], &g, sizeof(float));
        prm[(size_t)4 * i + 3] = stretch ? 1 : 0;
    }
    cudaStream_t st = (cudaStream_t)stream;
    double* scratch = nullptr;
    const size_t nd = (size_t)2 * n + (size_t)4 * n * w + h + (size_t)2 * n + 2;     // kx, ky, tables, params (4 ints = 2 doubles)
    HN_CUDA_OK(cudaMallocAsync(reinterpret_cast<void**>(&scratch), nd * sizeof(double), st));
    double* tables = scratch + 2 * (size_t)n;
    int* prm_dev = reinterpret_cast<int*>(tables + (size_t)4 * n * w + h);
    int rc = 0;
    if (cudaMemcpyAsync(scratch, k.data(), (size_t)2 * n * sizeof(double), cudaMemcpyHostToDevice, st) != cudaSuccess ||
        cudaMemcpyAsync(prm_dev, prm.data(), (size_t)4 * n * sizeof(int), cudaMemcpyHostToDevice, st) != cudaSuccess)
        rc = fail("hn_augment: parameter upload failed");
    // the host vectors are pageable: the runtime has staged them when cudaMemcpyAsync returns
    if (!rc) rc = augment_device(img, out, n, h, w, scratch, scratch + n, prm_dev, tables, st);
    cudaFreeAsync(scratch, st);
    return rc;
}

// ---- misc.pano_lsd_align.rotatePanorama (reference misc/pano_lsd_align.py:125-171) -------------------
int hn_rotate_panorama(const void* img, int in_is_f64, double* out, int n, int h, int w, int c, const double* rinv,
                       void* stream) {
    if (n == 0) return 0;
    HN_CHECK(img && out && rinv, "hn_rotate_panorama: NULL argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail("hn_rotate_panorama: no CUDA device -- libhorizonnet_b200 has no CPU path");
    return rotate_panorama_device(img, in_is_f64, out, n, h, w, c, rinv, (cudaStream_t)stream);
}

// ---- kernel-level entry points -----------------------------------------------------------------
int hn_conv2d(const float* in, int B, int H, int W, int Cin, int in_halo, const float* w, const float* scale,
              const float* shift, const float* residual, int Cout, int kh, int kw, int sh, int sw, int ph, int pw,
              int relu, float* out, int out_halo, int impl, void* stream) {
    HN_CHECK(in && w && scale && shift && out, "hn_conv2d: NULL argument");
    ConvDesc d;
    d.Cin = Cin; d.Cout = Cout; d.kh = kh; d.kw = kw; d.sh = sh; d.sw = sw; d.ph = ph; d.pw = pw; d.relu = relu;
    d.w = w; d.scale = scale; d.shift = shift;
    Act a = mk(const_cast<float*>(in), B, H, W, Cin, in_halo);
    const int Ho = (H + 2 * ph - kh) / sh + 1, Wo = (W + 2 * pw - kw) / sw + 1;
    Act o = mk(out, B, Ho, Wo, Cout, out_halo);
    if (impl == 1) {
        if (!conv_tc_supported(d, a, o)) return fail("hn_conv2d: shape not supported by the tcgen05 kernel");
        return conv_tc(d, a, o, residual, (cudaStream_t)stream);
    }
    return conv_f32(d, a, o, residual, (cudaStream_t)stream);
}

int hn_lstm_layer(const float* xproj, const float* whf, const float* whb, float* out, int T, int B, void* stream) {
    HN_CHECK(xproj && whf && whb && out && T >= 1 && B >= 1, "hn_lstm_layer: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    unsigned int* ctr = nullptr;
    HN_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&ctr), lstm_scratch_bytes()));
    int* flag = reinterpret_cast<int*>(ctr + 64);   // counters live in [0, 8), the error flag behind them (first KB of scratch)
    cudaMemsetAsync(ctr, 0, 1024, st);
    int rc = lstm_layer(xproj, whf, whb, out, T, B, ctr, flag, st);
    int h = 0;
    if (!rc) {
        if (cudaStreamSynchronize(st) != cudaSuccess) rc = fail("hn_lstm_layer: kernel failed");
        else {
            cudaMemcpy(&h, flag, sizeof(int), cudaMemcpyDeviceToHost);
            if (h) rc = fail("hn_lstm_layer: persistent kernel timed out waiting for a peer CTA");
        }
    }
    cudaFree(ctr);
    return rc;
}

}  // extern "C"
