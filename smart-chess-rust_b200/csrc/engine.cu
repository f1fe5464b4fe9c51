// sc_engine: weight loading / re-layout, device buffers, and the C ABI of include/sc_b200.h.
//
// One call of sc_eval() is the reference's `chess_tch_predict` (src/backends/torch.rs:89-146)
// for n leaves at once: H2D of the packed positions and legal moves, plane encode, the
// policy/value network, move-index gather + renormalisation, D2H of priors and values.
// There is no CPU fallback: without an sm_100 device sc_create() fails with SC_E_NOGPU.
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include <cuda_fp8.h>
#include <nvtx3/nvToolsExt.h>

#include "common.cuh"
#include "host/chess_rules.hpp"
#include "host/evaluator.hpp"
#include "host/host_util.hpp"

namespace scb {

// NVTX ranges around the phases of a call (visible in Nsight Systems / ncu --nvtx; no cost without a profiler
// attached).  The reference's hook for this is profiling/rocprof-selfplay:5-8.
struct NvtxRange {
    explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

static thread_local std::string g_err;
void set_error(const std::string &msg) { g_err = msg; }

struct Tensor {
    std::vector<uint32_t> dims;
    const float *data;
    size_t numel;
};

struct Blob {
    std::vector<char> raw;
    std::map<std::string, Tensor> t;
    int n_blocks = 0;
    // network variant (`NormTable`, `use_se`, py/module.py:6-9, 14-36), from the exporter's `__config__` tensor
    bool norm_folded = false;  // BatchNorm folded into conv weights + bias: the layers have no normalisation
    bool use_se = true;
};

static int read_blob(const char *path, Blob &b)
{
    FILE *f = fopen(path, "rb");
    if (!f) {
        set_error(std::string("cannot open weight blob: ") + path);
        return SC_E_IO;
    }
    fseek(f, 0, SEEK_END);
    long sz = ftell(f);
    fseek(f, 0, SEEK_SET);
    b.raw.resize((size_t)sz);
    size_t got = fread(b.raw.data(), 1, (size_t)sz, f);
    fclose(f);
    if (got != (size_t)sz || sz < 16 || memcmp(b.raw.data(), "SCB2WTS1", 8) != 0) {
        set_error("weight blob: bad magic or short read");
        return SC_E_IO;
    }
    const char *p = b.raw.data() + 8, *end = b.raw.data() + sz;
    auto rd32 = [&](uint32_t &v) { if (p + 4 > end) return false; memcpy(&v, p, 4); p += 4; return true; };
    auto rd64 = [&](uint64_t &v) { if (p + 8 > end) return false; memcpy(&v, p, 8); p += 8; return true; };
    uint32_t nb, nt;
    if (!rd32(nb) || !rd32(nt)) goto bad;
    b.n_blocks = (int)nb;
    struct Ent { std::string name; std::vector<uint32_t> dims; uint64_t off, numel; };
    {
        std::vector<Ent> ents(nt);
        for (uint32_t i = 0; i < nt; i++) {
            uint32_t nl, nd;
            if (!rd32(nl) || p + nl > end) goto bad;
            ents[i].name.assign(p, nl);
            p += nl;
            if (!rd32(nd) || nd > 8) goto bad;
            ents[i].dims.resize(nd);
            for (uint32_t d = 0; d < nd; d++)
                if (!rd32(ents[i].dims[d])) goto bad;
            if (!rd64(ents[i].off) || !rd64(ents[i].numel)) goto bad;
        }
        uint64_t data_bytes;
        if (!rd64(data_bytes) || p + data_bytes > end) goto bad;
        for (auto &e : ents) {
            if (e.off + e.numel * 4 > data_bytes) goto bad;
            b.t[e.name] = Tensor{e.dims, reinterpret_cast<const float *>(p + e.off), (size_t)e.numel};
        }
    }
    {
        auto it = b.t.find("__config__");
        if (it != b.t.end() && it->second.numel >= 2) {
            b.norm_folded = it->second.data[0] != 0.f;
            b.use_se = it->second.data[1] != 0.f;
        }
    }
    return SC_OK;
bad:
    set_error("weight blob: malformed header");
    return SC_E_IO;
}

static uint16_t f2bf(float f)
{
    uint32_t u;
    memcpy(&u, &f, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
    u += 0x7fffu + ((u >> 16) & 1u);  // round to nearest even
    return (uint16_t)(u >> 16);
}

// float -> fp16 bits, round to nearest even (subnormals kept, beyond the range +-inf)
static uint16_t f2h(float f)
{
    const __half h = __float2half_rn(f);
    uint16_t r;
    memcpy(&r, &h, 2);
    return r;
}

// The weights of a 16-bit tensor-core engine that become MMA / SE operands, rounded to its operand type.  An fp16 engine
// cannot represent a weight beyond +-65504: `bad` records one, and the load then fails naming the tensor (a bf16 engine
// has the fp32 exponent range and takes every finite weight).
struct Op16Weights {
    bool fp16;
    bool bad = false;
    uint16_t operator()(float f)
    {
        if (!fp16) return f2bf(f);
        if (fabsf(f) > 65504.f) bad = true;
        return f2h(f);
    }
    int check(const std::string &tensor) const
    {
        if (!bad) return SC_OK;
        set_error("weight blob: " + tensor + " has a weight beyond the fp16 range (|w| > 65504)");
        return SC_E_IO;
    }
};

// fp8 mode: the e4m3 weights of one output channel whose largest |w| is amax carry the scale s = 2^ceil(log2(amax / 448))
// (1 for an all-zero channel): w / s is at most 448 and is rounded to e4m3 (round to nearest even).  A power of two
// makes both w / s and the epilogue's acc * s exact, so the only rounding the scale brings is the operand's own.
static float e4m3_scale(float amax)
{
    if (!(amax > 0.f)) return 1.f;
    int e;
    const float f = frexpf(amax, &e);  // amax = f 2^e, f in [0.5, 1); 448 = 0.875 2^9
    return ldexpf(1.f, f <= 0.875f ? e - 9 : e - 8);
}
static uint8_t f2e4m3(float f) { return (uint8_t)__nv_cvt_float_to_fp8(f, __NV_SATFINITE, __NV_E4M3); }

// rows x k fp32 weights (row r at w[r * k], one output channel each) -> e4m3 bytes and the rows' scales
static void quantize_e4m3(const std::vector<float> &w, int rows, size_t k, std::vector<uint8_t> &q, std::vector<float> &scale)
{
    q.assign(w.size(), 0);
    scale.assign((size_t)rows, 1.f);
    for (int r = 0; r < rows; r++) {
        float amax = 0.f;
        for (size_t i = 0; i < k; i++) amax = fmaxf(amax, fabsf(w[r * k + i]));
        scale[r] = e4m3_scale(amax);
        for (size_t i = 0; i < k; i++) q[r * k + i] = f2e4m3(w[r * k + i] / scale[r]);
    }
}

struct ConvW {
    int taps = 1, cin = 0, cin_pad = 0, cout = 0, ldw = 0;
    float *w_f32 = nullptr;          // [taps][cin][ldw]        (fp32 mode)
    __nv_bfloat16 *w_bf16 = nullptr; // [taps][cout][cin_pad]   (tensor-core modes, K-major B operand; fp16 bits in fp16
                                     //                          mode, e4m3 bytes in fp8 mode)
    float *bias = nullptr, *gamma = nullptr, *beta = nullptr;
    float *scale = nullptr;          // fp8 mode: per output channel the weights' scale (e4m3_scale)
    TcConv *tc = nullptr;
};

struct SeW {
    float *w1t = nullptr, *b1 = nullptr, *w2t = nullptr, *b2 = nullptr;  // fp32 mode
    uint16_t *w1p = nullptr, *w2p = nullptr;                            // 16-bit modes, packed for the fused epilogue
    uint16_t *w1s[2] = {nullptr, nullptr}, *w2s[2] = {nullptr, nullptr};  // latency kernel: sliced per cluster rank (CL = 8, 4)
};

}  // namespace scb

using namespace scb;

struct sc_engine {
    int device = 0, mode = 0, max_batch = 0, n_blocks = 0, num_sms = 148;
    int mode_requested = 0;
    // SC_MODE_BF16 / SC_MODE_FP16 / SC_MODE_FP8: the same tensor-core kernels with bf16 / fp16 / e4m3 operands (tc_mode()
    // below).  fp8 has no latency kernel: every batch runs the throughput kernels
    TcOp op = TC_OP_BF16;
    // FP32 parity mode: the 256-wide convolutions as bf16x3 split GEMMs on the tensor cores (fp32 accumulate), LayerNorm /
    // SE / the narrow head layers in fp32 on the CUDA cores.  SC_MODE_FP32_FFMA = everything FFMA.
    bool fp32_tc = false;
    __nv_bfloat16 *p_x = nullptr, *p_t = nullptr;  // fp32_tc: activations as three bf16 planes [boards][64][768]
    int alloc_boards = 0;
    cudaStream_t stream = nullptr;
    std::vector<void *> allocs;
    ConvW stem;
    std::vector<ConvW> conv1, conv2;
    std::vector<SeW> se;
    ConvW pol1, pol2, val1;
    float *vfc_w_f32 = nullptr;           // fp32 mode: [16384][128]
    TcConv *vfc_tc = nullptr;             // bf16 mode: value FC as a split-K tcgen05 GEMM
    TcTower *tower = nullptr;             // bf16 mode: stem + all residual blocks in one launch
    LatTower *lat = nullptr;              // bf16 mode, small batches: the same layers, one 2-board tile per cluster
    int lat_max_boards = 0;
    // SCB200_LATENCY=0 keeps small batches on the throughput kernel (A/B runs and the bit-identity test)
    bool lat_enabled = !(getenv("SCB200_LATENCY") && getenv("SCB200_LATENCY")[0] == '0');
    double timed_flops_per_leaf = 0.0;    // FLOPs per leaf covered by the level-2 timed launches
    float *v_wmeta = nullptr, *v_b1 = nullptr, *v_w2 = nullptr, *v_b2 = nullptr;
    float *v_scale = nullptr;             // fp8 mode: the value FC's per-hidden-unit weight scales
    // io
    sc_position *d_pos = nullptr;
    sc_move *d_moves = nullptr;
    int32_t *d_off = nullptr;
    float *d_priors = nullptr, *d_value = nullptr, *d_meta = nullptr;
    int32_t *d_index = nullptr;
    int max_moves_total = 0;
    // activations
    float *f_planes = nullptr, *f_x = nullptr, *f_t = nullptr, *f_y = nullptr;
    __nv_bfloat16 *h_planes = nullptr, *h_x = nullptr, *h_t = nullptr, *h_y = nullptr;  // fp16 bits / e4m3 bytes
    float *logits = nullptr, *vpre = nullptr;
    int vsplit = 1;
    // gates
    void *d_scratch = nullptr;
    size_t scratch_bytes = 0;
    // accounting
    int64_t launches = 0;
    int timing = 0;
    // SCB200_FUSE_GATHER=0 keeps the stand-alone gather kernel (A/B runs)
    bool fuse_gather = !(getenv("SCB200_FUSE_GATHER") && getenv("SCB200_FUSE_GATHER")[0] == '0');
    // A/B switches, read when the engine is created: SCB200_TOWER=0 one launch per layer instead of the whole-tower
    // kernel; SCB200_TOWER_GROUP=n tiles per CTA carried through all layers together (0 = all)
    bool tower_enabled = !(getenv("SCB200_TOWER") && getenv("SCB200_TOWER")[0] == '0');
    int tower_group = getenv("SCB200_TOWER_GROUP") ? atoi(getenv("SCB200_TOWER_GROUP")) : 3;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    float last_tower_ms = 0.f, last_total_ms = 0.f;
    cudaEvent_t tickets[SC_MAX_INFLIGHT] = {nullptr, nullptr, nullptr, nullptr};
    int next_ticket = 0;
    int32_t *d_cnt = nullptr;
    unsigned int *d_vcount = nullptr;  // bf16 mode: arrival counters of the value FC's row tiles (value tail fused into the GEMM)
    // SCB200_FUSE_VALUE=0 keeps the stand-alone value_finish kernel (A/B runs)
    bool fuse_value = !(getenv("SCB200_FUSE_VALUE") && getenv("SCB200_FUSE_VALUE")[0] == '0');
    // asynchronous path (sc_eval_submit): two sets of device io buffers + copy streams, so the H2D of batch k+1
    // and the D2H of batch k-1 overlap the kernels of batch k
    struct IoSet {
        sc_position *pos = nullptr;
        sc_move *moves = nullptr;
        int32_t *cnt = nullptr;
        float *priors = nullptr, *value = nullptr;
        cudaEvent_t in_done = nullptr, compute_done = nullptr, out_done = nullptr;
    } io[2];
    cudaStream_t copy_in = nullptr, copy_out = nullptr;
    // small batches: the value head runs on its own stream next to the policy head (both are a few CTAs wide)
    cudaStream_t head_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    int64_t n_submits = 0;
    // small batches (sc_eval with n <= SC_SMALL_N): inputs are packed into ONE pinned staging buffer and travel in at
    // most one copy, the kernels write values + priors straight into another (a caller's Vec / numpy array is pageable
    // memory, which would otherwise make every one of the five copies a staged, blocking one)
    uint8_t *h_small_in = nullptr, *d_small_in = nullptr;
    float *h_small_out = nullptr;
    std::vector<cudaEvent_t> kev;  // level-2 timing: event pairs around the 3x3 256->256 convs
    int kev_used = 0;
    float last_conv_avg_ms = 0.f;
    int last_conv_n = 0;
    // sc_predict, set up by its first call: the legal-move kernel runs on gen_stream next to the encoder and the tower;
    // d_pred_out = [moves n x SC_MAX_MOVES | move counts n | termination codes n] for a call of n leaves, copied back
    // to h_pred_out in one piece
    cudaStream_t gen_stream = nullptr;
    cudaEvent_t ev_gen_fork = nullptr, ev_gen_done = nullptr;
    cudaEvent_t ev_gen_t[2] = {nullptr, nullptr};  // timing: around the legal-move kernel
    int8_t *d_pred_ep = nullptr;
    uint8_t *d_pred_out = nullptr, *h_pred_out = nullptr;
    float last_movegen_ms = 0.f;
    // sc_predict_stack, set up by its first call: stacks / offsets / n_hist of calls that do not fit the small staging
    // buffer, the replay's per-leaf status (copied back to h_replay_status) and its scratch, grown to the largest call
    sc_move *d_stack = nullptr;
    int32_t *d_stack_off = nullptr, *d_replay_status = nullptr, *h_replay_status = nullptr;
    int8_t *d_stack_nhist = nullptr;
    void *d_replay_scratch = nullptr;
    size_t replay_scratch_cap = 0;
    cudaEvent_t ev_replay_t[2] = {nullptr, nullptr};  // timing: around the replay kernel
    float last_replay_ms = 0.f;
    // sc_set_roots' table, set up by its first call: per root its final position and the offsets of its moves (device,
    // and a host copy in root_off), every root's replay records (grown to the largest call); n_roots == 0: no roots.
    // d_path_root: sc_predict_path's root indices of calls that do not fit the small staging buffer
    chess::Position *d_root_pos = nullptr;
    int32_t *d_root_off = nullptr, *d_path_root = nullptr;
    void *d_root_rec = nullptr;
    size_t root_rec_cap = 0;
    std::vector<int32_t> root_off;
    int n_roots = 0;
    float last_path_ms = 0.f;  // timing: the path-replay kernel (between ev_replay_t)
    // an sc_evaluator owns the stream: every other call that uses the device returns SC_E_STATE
    std::atomic<bool> evaluator{false};
};

namespace scb {

constexpr int SC_SMALL_N = 128;
// the pinned small-batch input buffer: sc_eval's positions, offsets and moves for SC_SMALL_N leaves
constexpr size_t SMALL_IN_BYTES = (size_t)SC_SMALL_N * (sizeof(sc_position) + 4 + SC_MAX_MOVES * sizeof(sc_move)) + 64;

// a tensor-core mode (bf16, fp16 or e4m3 operands): the tower and head kernels of tower_bf16.cu (and for the 16-bit
// types the latency kernel of tower_lat.cu)
static bool tc_mode(const sc_engine *e)
{
    return e->mode == SC_MODE_BF16 || e->mode == SC_MODE_FP16 || e->mode == SC_MODE_FP8;
}

template <typename T> static int dev_alloc(sc_engine *e, T **p, size_t count)
{
    void *q = nullptr;
    SCB_CUDA(cudaMalloc(&q, count * sizeof(T) + 256));
    SCB_CUDA(cudaMemset(q, 0, count * sizeof(T) + 256));
    e->allocs.push_back(q);
    *p = reinterpret_cast<T *>(q);
    return SC_OK;
}

template <typename T> static int upload(sc_engine *e, T **p, const std::vector<T> &h)
{
    SCB_CHECK(dev_alloc(e, p, h.size()));
    SCB_CUDA(cudaMemcpy(*p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
    return SC_OK;
}

static const Tensor *find(const Blob &b, const std::string &name)
{
    auto it = b.t.find(name);
    if (it == b.t.end()) {
        set_error("weight blob: missing tensor " + name);
        return nullptr;
    }
    return &it->second;
}

static int upload_vec(sc_engine *e, const Blob &b, const std::string &name, size_t expect, float **out)
{
    const Tensor *t = find(b, name);
    if (!t) return SC_E_IO;
    if (t->numel != expect) {
        set_error("weight blob: wrong size for " + name);
        return SC_E_IO;
    }
    std::vector<float> h(t->data, t->data + t->numel);
    return upload(e, out, h);
}

// conv weight [cout][cin][k][k] + bias + LayerNorm gamma/beta -> device layouts
static int load_conv(sc_engine *e, const Blob &b, const std::string &wname, const std::string &lnname, int taps,
                     int cin, int cout, ConvW &c, int epi = TC_EPI_LN)
{
    const Tensor *w = find(b, wname + ".weight");
    if (!w) return SC_E_IO;
    if (w->numel != (size_t)cout * cin * taps) {
        set_error("weight blob: wrong size for " + wname);
        return SC_E_IO;
    }
    c.taps = taps;
    c.cin = cin;
    c.cout = cout;
    c.cin_pad = (cin + 63) / 64 * 64;
    c.ldw = (cout + 127) / 128 * 128;
    SCB_CHECK(upload_vec(e, b, wname + ".bias", cout, &c.bias));
    if (!b.norm_folded) {  // folded BatchNorm: gamma == nullptr means "no normalisation" everywhere below
        SCB_CHECK(upload_vec(e, b, lnname + ".weight", cout, &c.gamma));
        SCB_CHECK(upload_vec(e, b, lnname + ".bias", cout, &c.beta));
    }
    if (e->mode == SC_MODE_FP32) {
        if (!(e->fp32_tc && cout == C_TOWER)) {
            std::vector<float> h((size_t)taps * cin * c.ldw, 0.f);
            for (int co = 0; co < cout; co++)
                for (int ci = 0; ci < cin; ci++)
                    for (int t = 0; t < taps; t++)
                        h[((size_t)t * cin + ci) * c.ldw + co] = w->data[((size_t)co * cin + ci) * taps + t];
            SCB_CHECK(upload(e, &c.w_f32, h));
        } else {
            // tensor-core parity mode: the weights' three bf16 planes side by side along K, [tap][cout][3 * cin_pad]
            const int kp = c.cin_pad;
            std::vector<uint16_t> h((size_t)taps * cout * 3 * kp, 0);
            for (int co = 0; co < cout; co++)
                for (int ci = 0; ci < cin; ci++)
                    for (int t = 0; t < taps; t++) {
                        float x = w->data[((size_t)co * cin + ci) * taps + t];
                        uint16_t *row = &h[((size_t)t * cout + co) * 3 * kp];
                        for (int pl = 0; pl < 3; pl++) {
                            const uint16_t b = f2bf(x);
                            row[pl * kp + ci] = b;
                            uint32_t u = (uint32_t)b << 16;
                            float back;
                            memcpy(&back, &u, 4);
                            x -= back;
                        }
                    }
            uint16_t *d = nullptr;
            SCB_CHECK(upload(e, &d, h));
            c.w_bf16 = reinterpret_cast<__nv_bfloat16 *>(d);
            SCB_CHECK(tc_split_conv_create(&c.tc, c.w_bf16, taps, kp, cin == C_IN ? 1 : 3, c.bias));
        }
    } else {
        // B operand, K-major: [tap][bn rows][cin_pad]; bn = 256, or 80 for the 73-wide policy conv
        const int bn = cout == C_TOWER ? C_TOWER : LD_POLICY;
        if (e->op == TC_OP_E4M3) {
            // per output channel [taps][cin_pad] -> e4m3 with the channel's scale, then [tap][bn][cin_pad]
            const size_t k = (size_t)taps * c.cin_pad;
            std::vector<float> wc((size_t)bn * k, 0.f);
            for (int co = 0; co < cout; co++)
                for (int ci = 0; ci < cin; ci++)
                    for (int t = 0; t < taps; t++) wc[co * k + (size_t)t * c.cin_pad + ci] = w->data[((size_t)co * cin + ci) * taps + t];
            std::vector<uint8_t> q, h(wc.size());
            std::vector<float> sc;
            quantize_e4m3(wc, bn, k, q, sc);
            for (int co = 0; co < bn; co++)
                for (int t = 0; t < taps; t++)
                    memcpy(&h[((size_t)t * bn + co) * c.cin_pad], &q[co * k + (size_t)t * c.cin_pad], (size_t)c.cin_pad);
            uint8_t *d = nullptr;
            SCB_CHECK(upload(e, &d, h));
            SCB_CHECK(upload(e, &c.scale, sc));
            c.w_bf16 = reinterpret_cast<__nv_bfloat16 *>(d);
            return tc_conv_create(&c.tc, c.w_bf16, taps, c.cin_pad, bn, epi, c.bias, c.gamma, c.beta, TC_OP_E4M3, c.scale);
        }
        std::vector<uint16_t> h((size_t)taps * bn * c.cin_pad, 0);
        Op16Weights cv{e->op == TC_OP_FP16};
        for (int co = 0; co < cout; co++)
            for (int ci = 0; ci < cin; ci++)
                for (int t = 0; t < taps; t++)
                    h[((size_t)t * bn + co) * c.cin_pad + ci] = cv(w->data[((size_t)co * cin + ci) * taps + t]);
        SCB_CHECK(cv.check(wname + ".weight"));
        uint16_t *d = nullptr;
        SCB_CHECK(upload(e, &d, h));
        c.w_bf16 = reinterpret_cast<__nv_bfloat16 *>(d);
        SCB_CHECK(tc_conv_create(&c.tc, c.w_bf16, taps, c.cin_pad, bn, epi, c.bias, c.gamma, c.beta, e->op));
    }
    return SC_OK;
}

static int load_weights(sc_engine *e, const Blob &b)
{
    e->n_blocks = b.n_blocks;
    SCB_CHECK(load_conv(e, b, "conv_block.0", "conv_block.1", 9, C_IN, C_TOWER, e->stem));
    e->conv1.resize(b.n_blocks);
    e->conv2.resize(b.n_blocks);
    e->se.resize(b.n_blocks);
    for (int i = 0; i < b.n_blocks; i++) {
        std::string p = "res_blocks." + std::to_string(i) + ".";
        SCB_CHECK(load_conv(e, b, p + "conv1", p + "bn1", 9, C_TOWER, C_TOWER, e->conv1[i]));
        SCB_CHECK(load_conv(e, b, p + "conv2", p + "bn2", 9, C_TOWER, C_TOWER, e->conv2[i], TC_EPI_LN_SE));
        if (!b.use_se) continue;  // residual-only blocks: out = relu(norm(conv2) + x)
        const Tensor *f1 = find(b, p + "se.fc1.weight"), *f2 = find(b, p + "se.fc2.weight");
        if (!f1 || !f2) return SC_E_IO;
        if (f1->numel != (size_t)C_SE * C_TOWER || f2->numel != (size_t)C_SE * C_TOWER) {
            set_error("weight blob: wrong SE size");
            return SC_E_IO;
        }
        std::vector<float> w1t((size_t)C_TOWER * C_SE), w2t((size_t)C_SE * C_TOWER);
        for (int j = 0; j < C_SE; j++)
            for (int c = 0; c < C_TOWER; c++) {
                w1t[(size_t)c * C_SE + j] = f1->data[(size_t)j * C_TOWER + c];
                w2t[(size_t)j * C_TOWER + c] = f2->data[(size_t)c * C_SE + j];
            }
        SCB_CHECK(upload_vec(e, b, p + "se.fc1.bias", C_SE, &e->se[i].b1));
        SCB_CHECK(upload_vec(e, b, p + "se.fc2.bias", C_TOWER, &e->se[i].b2));
        if (e->mode == SC_MODE_FP32) {
            SCB_CHECK(upload(e, &e->se[i].w1t, w1t));
            SCB_CHECK(upload(e, &e->se[i].w2t, w2t));
        } else {
            // packed so that epilogue thread j (fc1) / channel c (fc2) reads 8 consecutive inputs
            // with one coalesced 16-byte load: w1p[q][j][i] = fc1[j][8q+i], w2p[q][c][i] = fc2[c][8q+i]
            // (fp8 mode: bf16, the SE runs on the CUDA cores)
            std::vector<uint16_t> w1p((size_t)C_TOWER * C_SE), w2p((size_t)C_SE * C_TOWER);
            Op16Weights cv1{e->op == TC_OP_FP16}, cv2{e->op == TC_OP_FP16};
            for (int q = 0; q < C_TOWER / 8; q++)
                for (int j = 0; j < C_SE; j++)
                    for (int k = 0; k < 8; k++)
                        w1p[((size_t)q * C_SE + j) * 8 + k] = cv1(f1->data[(size_t)j * C_TOWER + 8 * q + k]);
            for (int q = 0; q < C_SE / 8; q++)
                for (int c = 0; c < C_TOWER; c++)
                    for (int k = 0; k < 8; k++)
                        w2p[((size_t)q * C_TOWER + c) * 8 + k] = cv2(f2->data[(size_t)c * C_SE + 8 * q + k]);
            SCB_CHECK(cv1.check(p + "se.fc1.weight"));
            SCB_CHECK(cv2.check(p + "se.fc2.weight"));
            SCB_CHECK(upload(e, &e->se[i].w1p, w1p));
            SCB_CHECK(upload(e, &e->se[i].w2p, w2p));
            // latency kernel: the same numbers sliced per cluster rank r -- fc1 COLUMNS (input channels) [r * NC, +NC)
            // for all 128 hidden units as [r][q][j][8], fc2 ROWS (output channels) [r * NC, +NC) as [r][q][c][8]
            for (int v = 0; v < 2; v++) {
                const int CL = v == 0 ? 8 : 4, NC = C_TOWER / CL;
                std::vector<uint16_t> a((size_t)C_TOWER * C_SE), b((size_t)C_SE * C_TOWER);
                for (int r = 0; r < CL; r++) {
                    for (int q = 0; q < NC / 8; q++)
                        for (int j = 0; j < C_SE; j++)
                            for (int k = 0; k < 8; k++)
                                a[(((size_t)r * (NC / 8) + q) * C_SE + j) * 8 + k] =
                                    cv1(f1->data[(size_t)j * C_TOWER + r * NC + 8 * q + k]);
                    for (int q = 0; q < C_SE / 8; q++)
                        for (int c = 0; c < NC; c++)
                            for (int k = 0; k < 8; k++)
                                b[(((size_t)r * (C_SE / 8) + q) * NC + c) * 8 + k] =
                                    cv2(f2->data[(size_t)(r * NC + c) * C_SE + 8 * q + k]);
                }
                SCB_CHECK(upload(e, &e->se[i].w1s[v], a));
                SCB_CHECK(upload(e, &e->se[i].w2s[v], b));
            }
            tc_conv_set_se(e->conv2[i].tc, e->se[i].w1p, e->se[i].b1, e->se[i].w2p, e->se[i].b2);
        }
    }
    SCB_CHECK(load_conv(e, b, "policy_head.model.0", "policy_head.model.1", 1, C_TOWER, C_TOWER, e->pol1));
    SCB_CHECK(load_conv(e, b, "policy_head.model.2", "policy_head.model.3", 1, C_TOWER, C_POLICY, e->pol2, TC_EPI_LN73));
    SCB_CHECK(load_conv(e, b, "value_head.conv.0", "value_head.conv.1", 1, C_TOWER, C_TOWER, e->val1));
    // value FC: [128][16391], columns c*64+s (NCHW flatten, py/module.py:93) then 7 meta
    const Tensor *fc = find(b, "value_head.ffn.0.weight");
    if (!fc) return SC_E_IO;
    const int KV = 64 * C_TOWER, KT = KV + SC_N_META;
    if (fc->numel != (size_t)N_VALUE_HIDDEN * KT) {
        set_error("weight blob: wrong value FC size");
        return SC_E_IO;
    }
    {
        std::vector<float> wm((size_t)SC_N_META * N_VALUE_HIDDEN);
        for (int j = 0; j < N_VALUE_HIDDEN; j++)
            for (int m = 0; m < SC_N_META; m++) wm[(size_t)m * N_VALUE_HIDDEN + j] = fc->data[(size_t)j * KT + KV + m];
        SCB_CHECK(upload(e, &e->v_wmeta, wm));
        // re-index K for NHWC activations: k' = s*256 + c  <-  k = c*64 + s
        if (e->mode == SC_MODE_FP32) {
            std::vector<float> h((size_t)KV * N_VALUE_HIDDEN);
            for (int j = 0; j < N_VALUE_HIDDEN; j++)
                for (int c = 0; c < C_TOWER; c++)
                    for (int s = 0; s < 64; s++)
                        h[((size_t)s * C_TOWER + c) * N_VALUE_HIDDEN + j] = fc->data[(size_t)j * KT + c * 64 + s];
            SCB_CHECK(upload(e, &e->vfc_w_f32, h));
        } else if (e->op == TC_OP_E4M3) {
            // the B operand below in e4m3, with the hidden units' scales
            std::vector<float> wf((size_t)N_VALUE_HIDDEN * KV);
            for (int j = 0; j < N_VALUE_HIDDEN; j++)
                for (int c = 0; c < C_TOWER; c++)
                    for (int s = 0; s < 64; s++) wf[(size_t)j * KV + (size_t)s * C_TOWER + c] = fc->data[(size_t)j * KT + c * 64 + s];
            std::vector<uint8_t> q;
            std::vector<float> sc;
            quantize_e4m3(wf, N_VALUE_HIDDEN, KV, q, sc);
            uint8_t *d = nullptr;
            SCB_CHECK(upload(e, &d, q));
            SCB_CHECK(upload(e, &e->v_scale, sc));
            SCB_CHECK(tc_conv_create(&e->vfc_tc, reinterpret_cast<__nv_bfloat16 *>(d), 1, KV, N_VALUE_HIDDEN, TC_EPI_RAW,
                                     nullptr, nullptr, nullptr, TC_OP_E4M3, e->v_scale));
        } else {
            // B operand of the value FC GEMM, K-major: [128][16384] with k' = s*256 + c
            // (the meta columns stay fp32: the fused value tail applies them)
            std::vector<uint16_t> h((size_t)N_VALUE_HIDDEN * KV);
            Op16Weights cv{e->op == TC_OP_FP16};
            for (int j = 0; j < N_VALUE_HIDDEN; j++)
                for (int c = 0; c < C_TOWER; c++)
                    for (int s = 0; s < 64; s++)
                        h[(size_t)j * KV + (size_t)s * C_TOWER + c] = cv(fc->data[(size_t)j * KT + c * 64 + s]);
            SCB_CHECK(cv.check("value_head.ffn.0.weight"));
            uint16_t *d = nullptr;
            SCB_CHECK(upload(e, &d, h));
            SCB_CHECK(tc_conv_create(&e->vfc_tc, reinterpret_cast<__nv_bfloat16 *>(d), 1, KV, N_VALUE_HIDDEN, TC_EPI_RAW,
                                     nullptr, nullptr, nullptr, e->op));
        }
    }
    SCB_CHECK(upload_vec(e, b, "value_head.ffn.0.bias", N_VALUE_HIDDEN, &e->v_b1));
    SCB_CHECK(upload_vec(e, b, "value_head.ffn.2.weight", N_VALUE_HIDDEN, &e->v_w2));
    SCB_CHECK(upload_vec(e, b, "value_head.ffn.2.bias", 1, &e->v_b2));
    return SC_OK;
}

static int alloc_buffers(sc_engine *e)
{
    const int B = (e->max_batch + 1) & ~1;
    e->alloc_boards = B;
    e->max_moves_total = e->max_batch * SC_MAX_MOVES;
    SCB_CHECK(dev_alloc(e, &e->d_pos, (size_t)B));
    SCB_CHECK(dev_alloc(e, &e->d_moves, (size_t)e->max_moves_total));
    SCB_CHECK(dev_alloc(e, &e->d_off, (size_t)B + 1));
    SCB_CHECK(dev_alloc(e, &e->d_cnt, (size_t)B + 1));
    SCB_CHECK(dev_alloc(e, &e->d_vcount, (size_t)(B + 127) / 128 + 1));  // zero-initialised by dev_alloc
    SCB_CHECK(dev_alloc(e, &e->d_priors, (size_t)e->max_moves_total));
    SCB_CHECK(dev_alloc(e, &e->d_index, (size_t)e->max_moves_total));
    SCB_CHECK(dev_alloc(e, &e->d_value, (size_t)B));
    SCB_CHECK(dev_alloc(e, &e->d_meta, (size_t)B * 8));
    SCB_CHECK(dev_alloc(e, &e->logits, (size_t)B * 64 * LD_POLICY));
    const size_t act = (size_t)B * 64 * C_TOWER;
    if (e->mode == SC_MODE_FP32) {
        e->vsplit = 16;  // the value FC has only n / 128 row tiles: split K over 16 CTAs each
        if (e->fp32_tc) {
            SCB_CHECK(dev_alloc(e, &e->h_planes, (size_t)B * 64 * C_IN_PAD));
            SCB_CHECK(dev_alloc(e, &e->p_x, act * 3));
            SCB_CHECK(dev_alloc(e, &e->p_t, act * 3));
        } else
            SCB_CHECK(dev_alloc(e, &e->f_planes, (size_t)B * 64 * C_IN));
        SCB_CHECK(dev_alloc(e, &e->f_x, act));
        SCB_CHECK(dev_alloc(e, &e->f_t, act));
        SCB_CHECK(dev_alloc(e, &e->f_y, act));
    } else {
        e->vsplit = 16;  // 16 k-blocks per work item: 16 CTAs share the 4 MB of value-FC weights even for one leaf
        SCB_CHECK(dev_alloc(e, &e->h_planes, (size_t)B * 64 * C_IN_PAD));
        SCB_CHECK(dev_alloc(e, &e->h_x, act));
        SCB_CHECK(dev_alloc(e, &e->h_t, act));
        SCB_CHECK(dev_alloc(e, &e->h_y, act));
    }
    SCB_CHECK(dev_alloc(e, &e->vpre, (size_t)e->vsplit * B * N_VALUE_HIDDEN));
    {
        const size_t in_bytes = SMALL_IN_BYTES;
        const size_t out_floats = (size_t)SC_SMALL_N * (1 + SC_MAX_MOVES);
        SCB_CHECK(dev_alloc(e, &e->d_small_in, in_bytes));
        SCB_CUDA(cudaMallocHost(&e->h_small_in, in_bytes));
        SCB_CUDA(cudaMallocHost(&e->h_small_out, out_floats * sizeof(float)));
    }
    // scratch for the gates: max(int8 planes + meta, fp32 NCHW planes + logp)
    e->scratch_bytes = (size_t)B * ((size_t)SC_N_PLANES * 64 * 4 + (size_t)SC_N_POLICY * 4 + 64);
    SCB_CHECK(dev_alloc(e, reinterpret_cast<char **>(&e->d_scratch), e->scratch_bytes));
    return SC_OK;
}

// level-2 timing: record the next event of the pair list on `st`
static int kev_mark(sc_engine *e, cudaStream_t st)
{
    if (e->timing < 2) return SC_OK;
    if (e->kev_used == (int)e->kev.size()) {
        cudaEvent_t ev;
        SCB_CUDA(cudaEventCreate(&ev));
        e->kev.push_back(ev);
    }
    SCB_CUDA(cudaEventRecord(e->kev[e->kev_used++], st));
    return SC_OK;
}

// the network on n boards; planes already in f_planes / h_planes, meta in d_meta.
// `gather` (16-bit modes only): the policy head's epilogue turns the logits into legal-move priors itself; the caller
// then skips launch_policy_gather.  Returns through *fused whether that happened.
// `gather_ready` (with `gather`): the policy head waits for this event first (sc_predict's legal moves)
static int run_network(sc_engine *e, int n, cudaStream_t st, const TcGather *gather = nullptr,
                       cudaEvent_t gather_ready = nullptr)
{
    NvtxRange nv_net("scb200: network (tower + heads)");
    const int rows = n * 64;
    e->kev_used = 0;
    if (e->timing) SCB_CUDA(cudaEventRecord(e->ev[1], st));
    if (e->mode == SC_MODE_FP32 && e->fp32_tc) {
        const int nb = e->alloc_boards;
        // 256-wide convolution: split GEMM on the tensor cores (fp32 out, + bias), then LayerNorm (+ReLU) in fp32;
        // `planes` = also emit the result as bf16x3 operand planes for the next convolution
        auto conv = [&](const ConvW &c, const __nv_bfloat16 *in, float *out, int relu, __nv_bfloat16 *planes, bool timed) -> int {
            if (timed) SCB_CHECK(kev_mark(e, st));
            SCB_CHECK(tc_conv_launch(c.tc, in, nb, n, out, nullptr, 0, 1, e->num_sms, st));
            if (timed) SCB_CHECK(kev_mark(e, st));
            SCB_CHECK(launch_ln_f32(out, rows, C_TOWER, C_TOWER, c.gamma, c.beta, relu, st, planes));
            e->launches += 2;
            return SC_OK;
        };
        SCB_CHECK(conv(e->stem, e->h_planes, e->f_x, 1, e->p_x, false));
        for (int i = 0; i < e->n_blocks; i++) {
            SCB_CHECK(conv(e->conv1[i], e->p_x, e->f_t, 1, e->p_t, true));
            SCB_CHECK(conv(e->conv2[i], e->p_t, e->f_y, 0, nullptr, true));
            SCB_CHECK(launch_se_res_f32(e->f_y, e->f_x, e->f_x, n, e->se[i].w1t, e->se[i].b1, e->se[i].w2t, e->se[i].b2, st,
                                        e->p_x));
            e->launches += 1;
        }
        e->timed_flops_per_leaf = 2.0 * 64 * 256 * 9.0 * 256 * 2 * e->n_blocks;
        if (e->timing) SCB_CUDA(cudaEventRecord(e->ev[2], st));
        SCB_CHECK(conv(e->pol1, e->p_x, e->f_t, 0, nullptr, false));
        SCB_CHECK(launch_gemm_f32(1, e->f_t, C_TOWER, e->pol2.w_f32, e->pol2.ldw, e->pol2.bias, e->logits, LD_POLICY,
                                  rows, C_POLICY, C_TOWER, st));
        SCB_CHECK(launch_ln_f32(e->logits, rows, C_POLICY, LD_POLICY, e->pol2.gamma, e->pol2.beta, 0, st));
        SCB_CHECK(conv(e->val1, e->p_x, e->f_y, 1, nullptr, false));
        SCB_CHECK(launch_gemm_f32(1, e->f_y, 64 * C_TOWER, e->vfc_w_f32, N_VALUE_HIDDEN, nullptr, e->vpre,
                                  N_VALUE_HIDDEN, n, N_VALUE_HIDDEN, 64 * C_TOWER, st, e->vsplit));
        e->launches += 3;
    } else if (e->mode == SC_MODE_FP32) {
        auto conv = [&](const ConvW &c, const float *in, int lda, float *out, int relu) -> int {
            SCB_CHECK(launch_gemm_f32(c.taps, in, lda, c.w_f32, c.ldw, c.bias, out, C_TOWER, rows, c.cout, c.cin, st));
            SCB_CHECK(launch_ln_f32(out, rows, c.cout, C_TOWER, c.gamma, c.beta, relu, st));
            e->launches += 2;
            return SC_OK;
        };
        SCB_CHECK(conv(e->stem, e->f_planes, C_IN, e->f_x, 1));
        for (int i = 0; i < e->n_blocks; i++) {
            SCB_CHECK(kev_mark(e, st));
            SCB_CHECK(launch_gemm_f32(9, e->f_x, C_TOWER, e->conv1[i].w_f32, e->conv1[i].ldw, e->conv1[i].bias, e->f_t,
                                      C_TOWER, rows, C_TOWER, C_TOWER, st));
            SCB_CHECK(kev_mark(e, st));
            SCB_CHECK(launch_ln_f32(e->f_t, rows, C_TOWER, C_TOWER, e->conv1[i].gamma, e->conv1[i].beta, 1, st));
            e->launches += 2;
            SCB_CHECK(kev_mark(e, st));
            SCB_CHECK(launch_gemm_f32(9, e->f_t, C_TOWER, e->conv2[i].w_f32, e->conv2[i].ldw, e->conv2[i].bias, e->f_y,
                                      C_TOWER, rows, C_TOWER, C_TOWER, st));
            SCB_CHECK(kev_mark(e, st));
            SCB_CHECK(launch_ln_f32(e->f_y, rows, C_TOWER, C_TOWER, e->conv2[i].gamma, e->conv2[i].beta, 0, st));
            e->launches += 2;
            SCB_CHECK(launch_se_res_f32(e->f_y, e->f_x, e->f_x, n, e->se[i].w1t, e->se[i].b1, e->se[i].w2t,
                                        e->se[i].b2, st));
            e->launches += 1;
        }
        if (e->timing) SCB_CUDA(cudaEventRecord(e->ev[2], st));
        // policy head
        SCB_CHECK(conv(e->pol1, e->f_x, C_TOWER, e->f_t, 0));
        SCB_CHECK(launch_gemm_f32(1, e->f_t, C_TOWER, e->pol2.w_f32, e->pol2.ldw, e->pol2.bias, e->logits, LD_POLICY,
                                  rows, C_POLICY, C_TOWER, st));
        SCB_CHECK(launch_ln_f32(e->logits, rows, C_POLICY, LD_POLICY, e->pol2.gamma, e->pol2.beta, 0, st));
        // value head
        SCB_CHECK(conv(e->val1, e->f_x, C_TOWER, e->f_y, 1));
        SCB_CHECK(launch_gemm_f32(1, e->f_y, 64 * C_TOWER, e->vfc_w_f32, N_VALUE_HIDDEN, nullptr, e->vpre,
                                  N_VALUE_HIDDEN, n, N_VALUE_HIDDEN, 64 * C_TOWER, st, e->vsplit));
        e->launches += 3;
    } else {
        const int nb = e->alloc_boards;
        int trc = SC_E_STATE;
        if (e->lat_enabled && e->lat && n <= e->lat_max_boards) {
            // small batch: one 2-board tile per cluster of 8 / 4 CTAs (same bits as the throughput kernel)
            SCB_CHECK(kev_mark(e, st));
            trc = lat_tower_launch(e->lat, n, st);
            if (trc == SC_OK) {
                SCB_CHECK(kev_mark(e, st));
                e->launches += 1;
                e->timed_flops_per_leaf =
                    2.0 * 64 * 256 * (9.0 * C_IN + e->n_blocks * (2 * 9.0 * 256 + 2.0 * C_SE / 64) + 2 * 256.0);
            } else if (trc != SC_E_STATE)
                return trc;
            else
                e->kev_used = 0;
        }
        if (trc != SC_OK && e->tower_enabled && e->tower) {
            SCB_CHECK(kev_mark(e, st));
            trc = tc_tower_launch(e->tower, n, e->num_sms, e->tower_group, st);
            if (trc == SC_OK) {
                SCB_CHECK(kev_mark(e, st));
                e->launches += 1;
                e->timed_flops_per_leaf =
                    2.0 * 64 * 256 * (9.0 * C_IN + e->n_blocks * (2 * 9.0 * 256 + 2.0 * C_SE / 64) + 2 * 256.0);
            } else if (trc != SC_E_STATE)
                return trc;
            else
                e->kev_used = 0;
        }
        if (trc != SC_OK) {
            SCB_CHECK(tc_conv_launch(e->stem.tc, e->h_planes, nb, n, e->h_x, nullptr, 1, 1, e->num_sms, st));
            e->launches += 1;
            for (int i = 0; i < e->n_blocks; i++) {
                SCB_CHECK(kev_mark(e, st));
                SCB_CHECK(tc_conv_launch(e->conv1[i].tc, e->h_x, nb, n, e->h_t, nullptr, 1, 1, e->num_sms, st));
                SCB_CHECK(kev_mark(e, st));
                SCB_CHECK(kev_mark(e, st));
                // conv2 + LN + squeeze-excitation + residual + ReLU, in place on the block input x
                SCB_CHECK(tc_conv_launch(e->conv2[i].tc, e->h_t, nb, n, e->h_x, e->h_x, 0, 1, e->num_sms, st));
                SCB_CHECK(kev_mark(e, st));
                e->launches += 2;
            }
            e->timed_flops_per_leaf = 2.0 * 64 * 256 * 9.0 * 256 * 2 * e->n_blocks;
        }
        if (e->timing) SCB_CUDA(cudaEventRecord(e->ev[2], st));
        NvtxRange nv_heads("scb200: policy + value heads");
        if (trc != SC_OK) {
            SCB_CHECK(tc_conv_launch(e->pol1.tc, e->h_x, nb, n, e->h_t, nullptr, 0, 1, e->num_sms, st));
            SCB_CHECK(tc_conv_launch(e->val1.tc, e->h_x, nb, n, e->h_y, nullptr, 1, 1, e->num_sms, st));
            e->launches += 2;
        }
        // one row tile (n <= 128): the value-FC GEMM finishes the value head itself (a launch is saved) and runs on its own
        // stream NEXT TO the policy head -- both are a few CTAs wide.  With more tiles the stand-alone tail kernel spreads
        // over the whole chip and is faster (28 vs 53 us at 2048), and the two heads each fill the chip.  Same bits either way.
        if (e->fuse_value && n <= 128) {
            const TcValueFinish vf{e->d_meta, e->v_wmeta, e->v_b1, e->v_w2, e->v_b2, e->d_value, e->d_vcount};
            if (!e->head_stream) {
                SCB_CUDA(cudaStreamCreateWithFlags(&e->head_stream, cudaStreamNonBlocking));
                SCB_CUDA(cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming));
                SCB_CUDA(cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming));
            }
            SCB_CUDA(cudaEventRecord(e->ev_fork, st));
            SCB_CUDA(cudaStreamWaitEvent(e->head_stream, e->ev_fork, 0));
            SCB_CHECK(tc_conv_launch(e->vfc_tc, e->h_y, nb, n, e->vpre, nullptr, 0, e->vsplit, e->num_sms, e->head_stream, nullptr, &vf));
            SCB_CUDA(cudaEventRecord(e->ev_join, e->head_stream));
            if (gather_ready) SCB_CUDA(cudaStreamWaitEvent(st, gather_ready, 0));
            SCB_CHECK(tc_conv_launch(e->pol2.tc, e->h_t, nb, n, e->logits, nullptr, 0, 1, e->num_sms, st, gather));
            SCB_CUDA(cudaStreamWaitEvent(st, e->ev_join, 0));
            e->launches += 2;
            return SC_OK;
        }
        if (gather_ready) SCB_CUDA(cudaStreamWaitEvent(st, gather_ready, 0));
        SCB_CHECK(tc_conv_launch(e->pol2.tc, e->h_t, nb, n, e->logits, nullptr, 0, 1, e->num_sms, st, gather));
        SCB_CHECK(tc_conv_launch(e->vfc_tc, e->h_y, nb, n, e->vpre, nullptr, 0, e->vsplit, e->num_sms, st));
        e->launches += 2;
    }
    SCB_CHECK(launch_value_finish(e->vpre, e->vsplit, n, e->d_meta, e->v_wmeta, e->v_b1, e->v_w2, e->v_b2,
                                  e->d_value, st, e->v_scale));
    e->launches += 1;
    return SC_OK;
}

static int encode_for_mode(sc_engine *e, const sc_position *d_pos, int n, cudaStream_t st)
{
    NvtxRange nv("scb200: encode planes");
    e->launches += 1;
    if (e->mode == SC_MODE_FP32 && !e->fp32_tc) return launch_encode_f32(d_pos, n, e->f_planes, e->d_meta, st);
    if (e->op == TC_OP_FP16) return launch_encode_fp16(d_pos, n, reinterpret_cast<__half *>(e->h_planes), e->d_meta, st);
    if (e->op == TC_OP_E4M3) return launch_encode_e4m3(d_pos, n, reinterpret_cast<uint8_t *>(e->h_planes), e->d_meta, st);
    return launch_encode_bf16(d_pos, n, e->h_planes, e->d_meta, st);
}

// sc_predict's buffers, stream and events (first call)
static int predict_setup(sc_engine *e)
{
    if (e->gen_stream) return SC_OK;
    const size_t out_b = (size_t)e->max_batch * (SC_MAX_MOVES * sizeof(sc_move) + 2 * sizeof(int32_t));
    SCB_CHECK(dev_alloc(e, &e->d_pred_ep, (size_t)e->max_batch));
    SCB_CHECK(dev_alloc(e, &e->d_pred_out, out_b));
    if (!e->h_pred_out) SCB_CUDA(cudaMallocHost(&e->h_pred_out, out_b));
    if (!e->ev_gen_fork) SCB_CUDA(cudaEventCreateWithFlags(&e->ev_gen_fork, cudaEventDisableTiming));
    if (!e->ev_gen_done) SCB_CUDA(cudaEventCreateWithFlags(&e->ev_gen_done, cudaEventDisableTiming));
    for (cudaEvent_t &ev : e->ev_gen_t)
        if (!ev) SCB_CUDA(cudaEventCreate(&ev));
    SCB_CUDA(cudaStreamCreateWithFlags(&e->gen_stream, cudaStreamNonBlocking));
    return SC_OK;
}

// grows *buf (*cap bytes) to hold the replay records of `positions` replayed positions; its contents are not kept
static int grow_records(void **buf, size_t *cap, int64_t positions)
{
    const size_t need = replay_scratch_bytes(positions);
    if (need > *cap) {
        if (*buf) SCB_CUDA(cudaFree(*buf));
        *buf = nullptr;
        *cap = 0;
        SCB_CUDA(cudaMalloc(buf, need));
        *cap = need;
    }
    return SC_OK;
}

// sc_predict_stack's buffers and events (first call), and a replay scratch for `positions` replayed positions
static int predict_stack_setup(sc_engine *e, int64_t positions)
{
    SCB_CHECK(predict_setup(e));
    if (!e->d_stack) {
        SCB_CHECK(dev_alloc(e, &e->d_stack, (size_t)e->max_batch * SC_MAX_STACK));
        SCB_CHECK(dev_alloc(e, &e->d_stack_off, (size_t)e->max_batch + 1));
        SCB_CHECK(dev_alloc(e, &e->d_stack_nhist, (size_t)e->max_batch));
        SCB_CHECK(dev_alloc(e, &e->d_replay_status, (size_t)e->max_batch));
        SCB_CUDA(cudaMallocHost(&e->h_replay_status, sizeof(int32_t) * (size_t)e->max_batch));
        for (cudaEvent_t &ev : e->ev_replay_t) SCB_CUDA(cudaEventCreate(&ev));
    }
    return grow_records(&e->d_replay_scratch, &e->replay_scratch_cap, positions);
}

// sc_set_roots' table (first call), with room for the records of `positions` replayed positions
static int roots_setup(sc_engine *e, int64_t positions)
{
    SCB_CHECK(predict_stack_setup(e, 0));
    if (!e->d_root_pos) {
        SCB_CHECK(dev_alloc(e, &e->d_root_pos, (size_t)e->max_batch));
        SCB_CHECK(dev_alloc(e, &e->d_root_off, (size_t)e->max_batch + 1));
        SCB_CHECK(dev_alloc(e, &e->d_path_root, (size_t)e->max_batch));
    }
    return grow_records(&e->d_root_rec, &e->root_rec_cap, positions);
}

// copies host arrays to the device on `st` and puts the address each is read from in dev[]: through the pinned small
// staging buffer in one copy when n <= SC_SMALL_N and they fit it, else each into its own device buffer.  Not read in
// place from pinned memory: the replay kernels read their moves one dependent ply at a time, each read a round trip
// over PCIe.  An input with no host array gets nullptr.
struct StagedInput {
    const void *src;
    size_t bytes;
    void *dev;  // its device buffer
};
static int stage_inputs(sc_engine *e, int n, std::initializer_list<StagedInput> in, const void **dev, cudaStream_t st)
{
    size_t total = 0;
    for (const StagedInput &a : in) total += a.bytes;
    const bool small = n <= SC_SMALL_N && total <= SMALL_IN_BYTES;
    size_t o = 0;
    for (const StagedInput &a : in) {
        if (small && a.bytes) memcpy(e->h_small_in + o, a.src, a.bytes);
        if (!small && a.bytes) SCB_CUDA(cudaMemcpyAsync(a.dev, a.src, a.bytes, cudaMemcpyHostToDevice, st));
        *dev++ = !a.src ? nullptr : small ? static_cast<const void *>(e->d_small_in + o) : a.dev;
        o += a.bytes;
    }
    if (small) SCB_CUDA(cudaMemcpyAsync(e->d_small_in, e->h_small_in, total, cudaMemcpyHostToDevice, st));
    return SC_OK;
}

// the host-side checks of n move lists (sc_predict_stack's stacks, sc_set_roots' roots, sc_predict_path's paths), before
// any launch: offsets off[0..n] from 0 and not decreasing, the game of list i -- base(i) plies stored before it, then its
// own -- at most SC_MAX_STACK plies, n_hist[i] (if given) in 1..min(SC_LOOKBACK, game plies + 1), every move's fields.
// `unit` names a list in the messages (list i as number first + i), `off_name` / `mv_name` the two arrays
template <class Base>
static int check_move_lists(const char *what, const char *unit, const char *off_name, const char *mv_name, int n,
                            const sc_move *mv, const int32_t *off, const int8_t *n_hist, Base base, int first = 0)
{
    const std::string w = std::string(what) + ": ";
    if (off[0] != 0) {
        set_error(w + off_name + "[0] = " + std::to_string(off[0]) + ", not 0");
        return SC_E_INVAL;
    }
    for (int i = 0; i < n; i++) {
        const int64_t own = (int64_t)off[i + 1] - off[i], len = base(i) + own;
        if (own < 0) {
            set_error(w + off_name + " decreases at " + unit + " " + std::to_string(first + i));
            return SC_E_INVAL;
        }
        if (len > SC_MAX_STACK) {
            set_error(w + unit + " " + std::to_string(first + i) + " has " + std::to_string(len) +
                      " plies, more than SC_MAX_STACK = " + std::to_string(SC_MAX_STACK));
            return SC_E_INVAL;
        }
        if (n_hist && (n_hist[i] < 1 || n_hist[i] > SC_LOOKBACK || n_hist[i] > len + 1)) {
            set_error(w + "n_hist[" + std::to_string(i) + "] = " + std::to_string(n_hist[i]) + " is not in 1.." +
                      std::to_string(len + 1 < SC_LOOKBACK ? len + 1 : SC_LOOKBACK));
            return SC_E_INVAL;
        }
    }
    const int total = off[n];
    if (total > 0 && !mv) {
        set_error(w + "bad argument");
        return SC_E_INVAL;
    }
    for (int k = 0; k < total; k++) {
        const sc_move m = mv[k];
        if (m.from >= 64 || m.to >= 64 || m.promo == 1 || m.promo > 5) {
            set_error(w + mv_name + "[" + std::to_string(k) + "] = (" + std::to_string(m.from) + ", " +
                      std::to_string(m.to) + ", " + std::to_string(m.promo) +
                      "): from/to must be below 64 and promo one of 0, 2, 3, 4, 5");
            return SC_E_INVAL;
        }
    }
    return SC_OK;
}

// the message of a replay status (REPLAY_STATUS)
static const char *replay_reason(int32_t status)
{
    static const char *why[] = {"", "its from-square holds no piece of the side to move",
                                "its to-square holds a piece of the side to move or a king",
                                "it promotes a piece that is not a pawn reaching the last rank",
                                "a pawn reaches the last rank without a promotion"};
    return why[status & 7];
}

// the message of a rejected replay: "<what>: <unit> <index>, ply <ply>: move rejected, <reason>"
static std::string replay_error(const char *what, const char *unit, int index, int ply, int32_t status)
{
    return std::string(what) + ": " + unit + " " + std::to_string(index) + ", ply " + std::to_string(ply) +
           ": move rejected, " + replay_reason(status);
}

// an evaluator's root slots (engine_backend_create): per slot SC_MAX_STACK + 1 replay records, the final position and
// the plies on the device, and the plies on the host (-1: the slot has no root)
struct SlotTable {
    void *d_rec = nullptr;
    chess::Position *d_pos = nullptr;
    int32_t *d_plies = nullptr;
    std::vector<int32_t> plies;
};

// SC_E_STATE while an evaluator owns the engine
static int check_owner(const sc_engine *e, const char *what)
{
    if (!e || !e->evaluator) return SC_OK;
    set_error(std::string(what) + ": the engine belongs to an evaluator until sc_evaluator_destroy");
    return SC_E_STATE;
}

static int finish_timing(sc_engine *e, cudaStream_t st)
{
    if (!e->timing) return SC_OK;
    SCB_CUDA(cudaEventRecord(e->ev[3], st));
    SCB_CUDA(cudaEventSynchronize(e->ev[3]));
    SCB_CUDA(cudaEventElapsedTime(&e->last_tower_ms, e->ev[1], e->ev[2]));
    SCB_CUDA(cudaEventElapsedTime(&e->last_total_ms, e->ev[0], e->ev[3]));
    if (e->timing >= 2) {
        float tot = 0.f;
        for (int i = 0; i + 1 < e->kev_used; i += 2) {
            float ms = 0.f;
            SCB_CUDA(cudaEventElapsedTime(&ms, e->kev[i], e->kev[i + 1]));
            tot += ms;
        }
        e->last_conv_n = e->kev_used / 2;
        e->last_conv_avg_ms = e->last_conv_n ? tot / e->last_conv_n : 0.f;
    }
    return SC_OK;
}

// sc_predict and sc_predict_stack once the packed leaves are on the device (d_pos / d_ep, as the kernels read them):
// the legal moves, the encoder, the network and the gather, and the copies back, all queued on `st`.  Up to
// SC_SMALL_N leaves write values and strided priors straight into the pinned small output buffer.
static int predict_launch(sc_engine *e, int n, const sc_position *d_pos, const int8_t *d_ep, float *priors_out,
                          float *value_out, cudaStream_t st)
{
    const size_t mv_b = sizeof(sc_move) * (size_t)n * SC_MAX_MOVES;
    const bool small = n <= SC_SMALL_N;
    float *d_value = small ? e->h_small_out : e->d_value, *d_priors = small ? e->h_small_out + n : e->d_priors;
    if (e->timing) SCB_CUDA(cudaEventRecord(e->ev[0], st));
    // the legal moves on their own stream next to the encoder and the tower (they do not depend on the network); the
    // policy head's gather waits for them
    sc_move *d_moves = reinterpret_cast<sc_move *>(e->d_pred_out);
    int32_t *d_cnt = reinterpret_cast<int32_t *>(e->d_pred_out + mv_b), *d_term = d_cnt + n;
    SCB_CUDA(cudaEventRecord(e->ev_gen_fork, st));
    SCB_CUDA(cudaStreamWaitEvent(e->gen_stream, e->ev_gen_fork, 0));
    if (e->timing) SCB_CUDA(cudaEventRecord(e->ev_gen_t[0], e->gen_stream));
    SCB_CHECK(launch_legal_moves(d_pos, d_ep, n, d_moves, d_cnt, d_term, e->gen_stream));
    if (e->timing) SCB_CUDA(cudaEventRecord(e->ev_gen_t[1], e->gen_stream));
    SCB_CUDA(cudaEventRecord(e->ev_gen_done, e->gen_stream));
    e->launches += 1;
    SCB_CHECK(encode_for_mode(e, d_pos, n, st));
    const TcGather g{d_pos, d_moves, nullptr, d_cnt, d_priors, n};
    const bool fused = tc_mode(e) && e->fuse_gather;
    float *saved_value = e->d_value;
    e->d_value = d_value;
    int rc = run_network(e, n, st, fused ? &g : nullptr, fused ? e->ev_gen_done : nullptr);
    e->d_value = saved_value;
    SCB_CHECK(rc);
    if (!fused) {
        SCB_CUDA(cudaStreamWaitEvent(st, e->ev_gen_done, 0));
        SCB_CHECK(launch_policy_gather(e->logits, d_pos, d_moves, nullptr, d_cnt, n, d_priors, st));
        e->launches += 1;
    }
    // results: moves, counts and termination codes in one copy, the full SC_MAX_MOVES stride of every leaf
    SCB_CUDA(cudaMemcpyAsync(e->h_pred_out, e->d_pred_out, mv_b + 2 * sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, st));
    if (!small) {
        SCB_CUDA(cudaMemcpyAsync(priors_out, d_priors, sizeof(float) * (size_t)n * SC_MAX_MOVES, cudaMemcpyDeviceToHost, st));
        SCB_CUDA(cudaMemcpyAsync(value_out, d_value, sizeof(float) * (size_t)n, cudaMemcpyDeviceToHost, st));
    }
    return SC_OK;
}

// waits for predict_launch's work and hands out its results; white(i): leaf i has White to move (for the terminal
// values)
template <class WhiteToMove>
static int predict_collect(sc_engine *e, const char *what, int n, sc_move *moves_out, int32_t *move_cnt_out,
                           float *priors_out, float *value_out, cudaStream_t st, WhiteToMove white)
{
    const size_t mv_b = sizeof(sc_move) * (size_t)n * SC_MAX_MOVES, cnt_b = sizeof(int32_t) * (size_t)n;
    const bool small = n <= SC_SMALL_N;
    SCB_CHECK(finish_timing(e, st));
    SCB_CUDA(cudaStreamSynchronize(st));
    if (e->timing) SCB_CUDA(cudaEventElapsedTime(&e->last_movegen_ms, e->ev_gen_t[0], e->ev_gen_t[1]));
    memcpy(moves_out, e->h_pred_out, mv_b);
    memcpy(move_cnt_out, e->h_pred_out + mv_b, cnt_b);
    if (small) {
        memcpy(value_out, e->h_small_out, sizeof(float) * (size_t)n);
        memcpy(priors_out, e->h_small_out + n, sizeof(float) * (size_t)n * SC_MAX_MOVES);
    }
    // a leaf without legal moves is terminal: torch.rs:98-106's value in White's perspective replaces the network's
    const int32_t *term = reinterpret_cast<const int32_t *>(e->h_pred_out + mv_b + cnt_b);
    int bad = -1;
    for (int i = 0; i < n; i++) {
        if (term[i] == PREDICT_OVERFLOW && bad < 0) bad = i;
        if (term[i] == chess::T_CHECKMATE) value_out[i] = white(i) ? -1.f : 1.f;
        if (term[i] == chess::T_STALEMATE) value_out[i] = 0.f;
    }
    if (bad >= 0) {
        set_error(std::string(what) + ": leaf " + std::to_string(bad) + " has more than " + std::to_string(SC_MAX_MOVES) +
                  " pseudo-legal moves (not a legal position)");
        return SC_E_INVAL;
    }
    return SC_OK;
}

// sc_predict_stack, sc_predict_path and an evaluator's pass after their own argument checks: leaf i is root root[i]
// of sc_set_roots' table or, with `slots`, of that slot table (root == nullptr: the initial position) followed by
// mv[off[i], off[i+1]).  The move lists' checks, the replay into d_pos /
// d_pred_ep, sc_predict's launches and the results.  off_name / mv_name: the two arrays in messages; replay_ms: where
// timing puts the replay kernel's time
static int predict_replay(sc_engine *e, const char *what, int n, const int32_t *root, const SlotTable *slots,
                          const sc_move *mv, const int32_t *off, const char *off_name, const char *mv_name,
                          const int8_t *n_hist, sc_position *pos_out, sc_move *moves_out, int32_t *move_cnt_out,
                          float *priors_out, float *value_out, float *replay_ms, void *stream)
{
    const int32_t *ro = e->root_off.data();
    auto root_plies = [&](int i) {
        return !root ? 0 : slots ? slots->plies[root[i]] : ro[root[i] + 1] - ro[root[i]];
    };
    SCB_CHECK(check_move_lists(what, "leaf", off_name, mv_name, n, mv, off, n_hist, root_plies));
    cudaStream_t st = stream ? (cudaStream_t)stream : e->stream;
    SCB_CUDA(cudaSetDevice(e->device));
    const int total = off[n];
    SCB_CHECK(predict_stack_setup(e, (int64_t)total + n));
    const void *d[4];
    SCB_CHECK(stage_inputs(e, n,
                           {{off, sizeof(int32_t) * ((size_t)n + 1), e->d_stack_off},
                            {root, root ? sizeof(int32_t) * (size_t)n : 0, e->d_path_root},
                            {mv, sizeof(sc_move) * (size_t)total, e->d_stack},
                            {n_hist, n_hist ? (size_t)n : 0, e->d_stack_nhist}},
                           d, st));
    // the packed leaves and their ep squares go where sc_predict's kernels read them on the device
    if (e->timing) SCB_CUDA(cudaEventRecord(e->ev_replay_t[0], st));
    SCB_CHECK(launch_path_replay(slots ? slots->d_rec : e->d_root_rec, e->d_root_off, slots ? slots->d_plies : nullptr,
                                 slots ? slots->d_pos : e->d_root_pos, static_cast<const int32_t *>(d[1]),
                                 static_cast<const sc_move *>(d[2]), static_cast<const int32_t *>(d[0]),
                                 static_cast<const int8_t *>(d[3]), n, e->d_replay_scratch, e->d_pos, e->d_pred_ep,
                                 e->d_replay_status, st));
    if (e->timing) SCB_CUDA(cudaEventRecord(e->ev_replay_t[1], st));
    e->launches += 1;
    SCB_CHECK(predict_launch(e, n, e->d_pos, e->d_pred_ep, priors_out, value_out, st));
    SCB_CUDA(cudaMemcpyAsync(e->h_replay_status, e->d_replay_status, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, st));
    if (pos_out) SCB_CUDA(cudaMemcpyAsync(pos_out, e->d_pos, sizeof(sc_position) * (size_t)n, cudaMemcpyDeviceToHost, st));
    // the side to move of a leaf replayed from the initial position: White after an even number of plies
    const int32_t *status = e->h_replay_status;
    auto plies = [&](int i) { return status[i] ? status[i] >> 3 : root_plies(i) + off[i + 1] - off[i]; };
    const int rc = predict_collect(e, what, n, moves_out, move_cnt_out, priors_out, value_out, st,
                                   [&](int i) { return plies(i) % 2 == 0; });
    if (rc != SC_OK && rc != SC_E_INVAL) return rc;
    if (e->timing) SCB_CUDA(cudaEventElapsedTime(replay_ms, e->ev_replay_t[0], e->ev_replay_t[1]));
    for (int i = 0; i < n; i++) {
        if (!status[i]) continue;
        set_error(replay_error(what, "leaf", i, plies(i), status[i]));
        return SC_E_INVAL;
    }
    return rc;
}

// the engine behind an sc_evaluator (host/evaluator.hpp): its slot table, the root updates' launch, and each pass of
// leaves through predict_replay.  The dispatcher thread is the only caller
class EngineBackend : public EvalBackend {
    sc_engine *e_;
    SlotTable t_;
    // one pass: the requests that passed their checks, as predict_replay / launch_slot_replay take them
    std::vector<int32_t> root_, off_;
    std::vector<sc_move> mv_;
    std::vector<int8_t> flag_;  // update: append; leaf: n_hist
    std::vector<sc_position> pos_;
    std::vector<sc_move> moves_;
    std::vector<int32_t> cnt_;
    std::vector<float> priors_, value_;

    void clear()
    {
        root_.clear();
        off_.assign(1, 0);
        mv_.clear();
        flag_.clear();
    }
    void add(int slot, const sc_move *mv, int len, int8_t flag)
    {
        root_.push_back(slot);
        mv_.insert(mv_.end(), mv, mv + len);
        off_.push_back((int32_t)mv_.size());
        flag_.push_back(flag);
    }
    // the updates' one launch; statuses in e_->h_replay_status
    int launch_updates(int n)
    {
        cudaStream_t st = e_->stream;
        SCB_CUDA(cudaSetDevice(e_->device));
        const void *d[4];
        SCB_CHECK(stage_inputs(e_, n,
                               {{off_.data(), sizeof(int32_t) * ((size_t)n + 1), e_->d_stack_off},
                                {root_.data(), sizeof(int32_t) * (size_t)n, e_->d_path_root},
                                {flag_.data(), (size_t)n, e_->d_stack_nhist},
                                {mv_.data(), sizeof(sc_move) * mv_.size(), e_->d_stack}},
                               d, st));
        SCB_CHECK(launch_slot_replay(static_cast<const sc_move *>(d[3]), static_cast<const int32_t *>(d[0]),
                                     static_cast<const int32_t *>(d[1]), static_cast<const int8_t *>(d[2]), n, t_.d_rec,
                                     t_.d_pos, t_.d_plies, e_->d_replay_status, st));
        e_->launches += 1;
        SCB_CUDA(cudaMemcpyAsync(e_->h_replay_status, e_->d_replay_status, sizeof(int32_t) * (size_t)n,
                                 cudaMemcpyDeviceToHost, st));
        SCB_CUDA(cudaStreamSynchronize(st));
        return SC_OK;
    }

public:
    explicit EngineBackend(sc_engine *e) : e_(e) {}
    ~EngineBackend() override
    {
        cudaSetDevice(e_->device);
        cudaStreamSynchronize(e_->stream);
        if (t_.d_rec) cudaFree(t_.d_rec);
        if (t_.d_pos) cudaFree(t_.d_pos);
        if (t_.d_plies) cudaFree(t_.d_plies);
        e_->evaluator = false;
    }
    int setup(int n_slots)
    {
        SCB_CUDA(cudaSetDevice(e_->device));
        SCB_CHECK(roots_setup(e_, 0));  // the staging buffers of sc_set_roots / sc_predict_path
        SCB_CUDA(cudaMalloc(&t_.d_rec, replay_scratch_bytes((int64_t)n_slots * (SC_MAX_STACK + 1))));
        SCB_CUDA(cudaMalloc(&t_.d_pos, sizeof(chess::Position) * (size_t)n_slots));
        SCB_CUDA(cudaMalloc(&t_.d_plies, sizeof(int32_t) * (size_t)n_slots));
        t_.plies.assign((size_t)n_slots, -1);
        return SC_OK;
    }

    void update_roots(const std::vector<RootUpdate *> &u) override
    {
        std::vector<RootUpdate *> run;
        clear();
        for (RootUpdate *r : u) {
            const char *what = r->append ? "sc_evaluator_extend_root" : "sc_evaluator_set_root";
            const int ply0 = r->append ? t_.plies[r->slot] : 0;
            if (ply0 < 0) {
                r->rc = SC_E_STATE;
                r->err = std::string(what) + ": slot " + std::to_string(r->slot) + " has no root";
                continue;
            }
            const int32_t off[2] = {0, r->len};
            r->rc = check_move_lists(what, "slot", "len", r->append ? "moves" : "stack", 1, r->moves, off, nullptr,
                                     [&](int) { return ply0; }, r->slot);
            if (r->rc != SC_OK) {
                r->err = g_err;
                continue;
            }
            run.push_back(r);
            add(r->slot, r->moves, r->len, r->append);
        }
        if (run.empty()) return;
        const int rc = launch_updates((int)run.size());
        for (size_t i = 0; i < run.size(); i++) {
            RootUpdate *r = run[i];
            const int32_t status = e_->h_replay_status[i];
            const int ply0 = r->append ? t_.plies[r->slot] : 0;
            if (rc != SC_OK || status) {
                r->rc = rc != SC_OK ? rc : SC_E_INVAL;
                r->err = rc != SC_OK ? g_err
                                     : replay_error(r->append ? "sc_evaluator_extend_root" : "sc_evaluator_set_root",
                                                    "slot", r->slot, status >> 3, status);
                t_.plies[r->slot] = -1;
            } else {
                t_.plies[r->slot] = ply0 + r->len;
            }
        }
    }

    void predict(const std::vector<LeafRequest *> &req) override
    {
        const char *what = "sc_evaluator_predict";
        std::vector<LeafRequest *> run;
        bool want_pos = false;
        clear();
        for (LeafRequest *q : req) {
            const int plies = t_.plies[q->slot];
            if (plies < 0) {
                q->rc = SC_E_STATE;
                q->err = std::string(what) + ": slot " + std::to_string(q->slot) + " has no root (sc_evaluator_set_root)";
                continue;
            }
            if (q->n_hist < 0 || q->n_hist > SC_LOOKBACK) {
                q->rc = SC_E_INVAL;
                q->err = std::string(what) + ": n_hist = " + std::to_string(q->n_hist) + " is not in 0..8";
                continue;
            }
            const int32_t off[2] = {0, q->len};
            const int8_t nh = (int8_t)q->n_hist;
            q->rc = check_move_lists(what, "slot", "len", "path", 1, q->path, off, nh ? &nh : nullptr,
                                     [&](int) { return plies; }, q->slot);
            if (q->rc != SC_OK) {
                q->err = g_err;
                continue;
            }
            const int total = plies + q->len;
            run.push_back(q);
            add(q->slot, q->path, q->len, nh ? nh : (int8_t)(total + 1 < SC_LOOKBACK ? total + 1 : SC_LOOKBACK));
            want_pos |= q->pos_out != nullptr;
        }
        if (run.empty()) return;
        const size_t n = run.size();
        if (moves_.size() < n * SC_MAX_MOVES) {
            pos_.resize(n);
            moves_.resize(n * SC_MAX_MOVES);
            cnt_.resize(n);
            priors_.resize(n * SC_MAX_MOVES);
            value_.resize(n);
        }
        float replay_ms = 0.f;
        const int rc = predict_replay(e_, what, (int)n, root_.data(), &t_, mv_.data(), off_.data(), "len", "path",
                                      flag_.data(), want_pos ? pos_.data() : nullptr, moves_.data(), cnt_.data(),
                                      priors_.data(), value_.data(), &replay_ms, nullptr);
        // a rejected leaf fails its own caller (the replay's status, the move generator's termination code)
        const int32_t *status = e_->h_replay_status;
        const int32_t *term = reinterpret_cast<const int32_t *>(e_->h_pred_out + (sizeof(sc_move) * SC_MAX_MOVES +
                                                                                  sizeof(int32_t)) * n);
        for (size_t i = 0; i < n; i++) {
            LeafRequest *q = run[i];
            if (rc != SC_OK && rc != SC_E_INVAL) {
                q->rc = rc;
                q->err = g_err;
                continue;
            }
            memcpy(q->moves_out, &moves_[i * SC_MAX_MOVES], sizeof(sc_move) * SC_MAX_MOVES);
            memcpy(q->priors_out, &priors_[i * SC_MAX_MOVES], sizeof(float) * SC_MAX_MOVES);
            *q->move_cnt_out = cnt_[i];
            *q->value_out = value_[i];
            if (q->pos_out) *q->pos_out = pos_[i];
            if (status[i]) {
                q->rc = SC_E_INVAL;
                q->err = replay_error(what, "slot", q->slot, status[i] >> 3, status[i]);
            } else if (term[i] == PREDICT_OVERFLOW) {
                q->rc = SC_E_INVAL;
                q->err = std::string(what) + ": slot " + std::to_string(q->slot) + " has more than " +
                         std::to_string(SC_MAX_MOVES) + " pseudo-legal moves (not a legal position)";
            }
        }
    }
};

int engine_backend_create(sc_engine *e, int n_slots, int *max_batch, EvalBackend **out)
{
    if (!e || n_slots < 1 || n_slots > e->max_batch) {
        set_error("sc_evaluator_create: bad argument (n_slots must be in 1..max_batch)");
        return SC_E_INVAL;
    }
    bool free_engine = false;
    if (!e->evaluator.compare_exchange_strong(free_engine, true)) {
        set_error("sc_evaluator_create: the engine already has an evaluator");
        return SC_E_STATE;
    }
    EngineBackend *b = new EngineBackend(e);  // gives the engine back when deleted
    const int rc = b->setup(n_slots);
    if (rc != SC_OK) {
        const std::string msg = g_err;
        delete b;
        set_error(msg);
        return rc;
    }
    *max_batch = e->max_batch;
    *out = b;
    return SC_OK;
}

}  // namespace scb

extern "C" {

const char *sc_last_error(void) { return g_err.c_str(); }

int sc_create(const char *weights_blob_path, int device, int mode, int max_batch, sc_engine **out)
{
    if (!out || !weights_blob_path || max_batch <= 0 ||
        (mode != SC_MODE_FP32 && mode != SC_MODE_BF16 && mode != SC_MODE_FP32_FFMA && mode != SC_MODE_FP16 &&
         mode != SC_MODE_FP8)) {
        set_error("sc_create: bad argument");
        return SC_E_INVAL;
    }
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device >= ndev) {
        set_error("sc_create: no CUDA device (this backend has no CPU fallback)");
        return SC_E_NOGPU;
    }
    cudaDeviceProp prop;
    SCB_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        set_error("sc_create: device is not sm_100 (Blackwell B200); kernels are built for sm_100a only");
        return SC_E_NOGPU;
    }
    SCB_CUDA(cudaSetDevice(device));
    Blob blob;
    SCB_CHECK(read_blob(weights_blob_path, blob));
    sc_engine *e = new sc_engine();
    e->device = device;
    e->mode_requested = mode;
    e->mode = mode == SC_MODE_FP32_FFMA ? SC_MODE_FP32 : mode;
    e->fp32_tc = mode == SC_MODE_FP32;
    e->op = mode == SC_MODE_FP16 ? TC_OP_FP16 : mode == SC_MODE_FP8 ? TC_OP_E4M3 : TC_OP_BF16;
    e->max_batch = max_batch;
    e->num_sms = prop.multiProcessorCount;
    int rc = SC_OK;
    do {
        if (cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) != cudaSuccess) { rc = SC_E_CUDA; set_error("stream create failed"); break; }
        for (int i = 0; i < 4; i++)
            if (cudaEventCreate(&e->ev[i]) != cudaSuccess) { rc = SC_E_CUDA; set_error("event create failed"); break; }
        if (rc) break;
        if ((rc = load_weights(e, blob)) != SC_OK) break;
        if ((rc = alloc_buffers(e)) != SC_OK) break;
        if ((rc = upload_move_tables(e->stream)) != SC_OK) break;
        if (tc_mode(e)) {
            std::vector<TcTowerLayerDesc> d;
            d.push_back(TcTowerLayerDesc{e->stem.tc, e->h_planes, e->h_x, nullptr, 1});
            for (int i = 0; i < e->n_blocks; i++) {
                d.push_back(TcTowerLayerDesc{e->conv1[i].tc, e->h_x, e->h_t, nullptr, 1});
                d.push_back(TcTowerLayerDesc{e->conv2[i].tc, e->h_t, e->h_x, e->h_x, 0});
            }
            // the two 256-wide 1x1 head convolutions read the tower output tile by tile as well
            d.push_back(TcTowerLayerDesc{e->pol1.tc, e->h_x, e->h_t, nullptr, 0});
            d.push_back(TcTowerLayerDesc{e->val1.tc, e->h_x, e->h_y, nullptr, 1});
            if ((rc = tc_tower_create(&e->tower, d.data(), (int)d.size(), e->alloc_boards, e->op)) != SC_OK) break;
            // the same layers for the latency kernel (fp8 is a throughput mode: it has none)
            if (e->op != TC_OP_E4M3) {
                std::vector<LatLayerDesc> ld;
                auto lat_layer = [&](const ConvW &c, const __nv_bfloat16 *in, void *out, const __nv_bfloat16 *resid, int relu,
                                     int se, const SeW *sw) {
                    LatLayerDesc L{};
                    L.w = c.w_bf16;
                    L.taps = c.taps;
                    L.cin_pad = c.cin_pad;
                    L.in = in;
                    L.out = out;
                    L.resid = resid;
                    L.bias = c.bias;
                    L.gamma = c.gamma;
                    L.beta = c.beta;
                    L.relu = relu;
                    L.ln = c.gamma != nullptr;
                    L.se = se;
                    if (sw) {
                        L.se_w1s8 = sw->w1s[0];
                        L.se_w2s8 = sw->w2s[0];
                        L.se_w1s4 = sw->w1s[1];
                        L.se_w2s4 = sw->w2s[1];
                        L.se_b1 = sw->b1;
                        L.se_b2 = sw->b2;
                    }
                    ld.push_back(L);
                };
                lat_layer(e->stem, e->h_planes, e->h_x, nullptr, 1, 0, nullptr);
                for (int i = 0; i < e->n_blocks; i++) {
                    lat_layer(e->conv1[i], e->h_x, e->h_t, nullptr, 1, 0, nullptr);
                    const bool has_se = e->se[i].w1p != nullptr;
                    lat_layer(e->conv2[i], e->h_t, e->h_x, e->h_x, 0, has_se ? 1 : 2, has_se ? &e->se[i] : nullptr);
                }
                lat_layer(e->pol1, e->h_x, e->h_t, nullptr, 0, 0, nullptr);
                lat_layer(e->val1, e->h_x, e->h_y, nullptr, 1, 0, nullptr);
                if ((rc = lat_tower_create(&e->lat, ld.data(), (int)ld.size(), e->alloc_boards, e->op == TC_OP_FP16)) != SC_OK) break;
                e->lat_max_boards = lat_tower_max_boards(e->lat);
            }
        }
        if (cudaDeviceSynchronize() != cudaSuccess) { rc = SC_E_CUDA; set_error("sync after weight upload failed"); break; }
    } while (0);
    if (rc != SC_OK) {
        sc_destroy(e);
        return rc;
    }
    *out = e;
    return SC_OK;
}

int sc_destroy(sc_engine *e)
{
    if (!e) return SC_OK;
    SCB_CHECK(check_owner(e, "sc_destroy"));
    cudaSetDevice(e->device);
    cudaDeviceSynchronize();
    auto kill = [](ConvW &c) { if (c.tc) tc_conv_destroy(c.tc); c.tc = nullptr; };
    kill(e->stem); kill(e->pol1); kill(e->pol2); kill(e->val1);
    if (e->vfc_tc) tc_conv_destroy(e->vfc_tc);
    if (e->tower) tc_tower_destroy(e->tower);
    if (e->lat) lat_tower_destroy(e->lat);
    for (auto &c : e->conv1) kill(c);
    for (auto &c : e->conv2) kill(c);
    for (void *p : e->allocs) cudaFree(p);
    if (e->h_small_in) cudaFreeHost(e->h_small_in);
    if (e->h_small_out) cudaFreeHost(e->h_small_out);
    for (int i = 0; i < 4; i++)
        if (e->ev[i]) cudaEventDestroy(e->ev[i]);
    for (cudaEvent_t ev : e->kev) cudaEventDestroy(ev);
    for (int i = 0; i < SC_MAX_INFLIGHT; i++)
        if (e->tickets[i]) cudaEventDestroy(e->tickets[i]);
    for (auto &s : e->io) {
        if (s.in_done) cudaEventDestroy(s.in_done);
        if (s.compute_done) cudaEventDestroy(s.compute_done);
        if (s.out_done) cudaEventDestroy(s.out_done);
    }
    if (e->h_pred_out) cudaFreeHost(e->h_pred_out);
    if (e->h_replay_status) cudaFreeHost(e->h_replay_status);
    if (e->d_replay_scratch) cudaFree(e->d_replay_scratch);
    if (e->d_root_rec) cudaFree(e->d_root_rec);
    for (cudaEvent_t ev : {e->ev_gen_fork, e->ev_gen_done, e->ev_gen_t[0], e->ev_gen_t[1], e->ev_replay_t[0], e->ev_replay_t[1]})
        if (ev) cudaEventDestroy(ev);
    if (e->gen_stream) cudaStreamDestroy(e->gen_stream);
    if (e->head_stream) cudaStreamDestroy(e->head_stream);
    if (e->ev_fork) cudaEventDestroy(e->ev_fork);
    if (e->ev_join) cudaEventDestroy(e->ev_join);
    if (e->copy_in) cudaStreamDestroy(e->copy_in);
    if (e->copy_out) cudaStreamDestroy(e->copy_out);
    if (e->stream) cudaStreamDestroy(e->stream);
    delete e;
    return SC_OK;
}

int sc_info(const sc_engine *e, int *n_res_blocks, int *max_batch, int *mode)
{
    if (!e) return SC_E_INVAL;
    if (n_res_blocks) *n_res_blocks = e->n_blocks;
    if (max_batch) *max_batch = e->max_batch;
    if (mode) *mode = e->mode_requested;
    return SC_OK;
}

int sc_device_info(const sc_engine *e, int *device, int *num_sms)
{
    if (!e) return SC_E_INVAL;
    if (device) *device = e->device;
    if (num_sms) *num_sms = e->num_sms;
    return SC_OK;
}

int sc_eval_device(sc_engine *e, int n, const void *d_pos, const void *d_moves, const void *d_move_off,
                   int n_moves_total, void *d_priors_out, void *d_value_out, void *stream)
{
    SCB_CHECK(check_owner(e, "sc_eval_device"));
    if (!e || n < 0 || n > e->max_batch) {
        set_error("sc_eval_device: bad n");
        return SC_E_INVAL;
    }
    (void)n_moves_total;
    if (n == 0) return SC_OK;
    cudaStream_t st = stream ? (cudaStream_t)stream : e->stream;
    SCB_CUDA(cudaSetDevice(e->device));
    if (e->timing) SCB_CUDA(cudaEventRecord(e->ev[0], st));
    const sc_position *pos = static_cast<const sc_position *>(d_pos);
    SCB_CHECK(encode_for_mode(e, pos, n, st));
    // value goes straight to the caller's buffer
    float *saved = e->d_value;
    e->d_value = static_cast<float *>(d_value_out);
    const TcGather g{pos, static_cast<const sc_move *>(d_moves), static_cast<const int32_t *>(d_move_off), nullptr,
                     static_cast<float *>(d_priors_out), n};
    const bool fused = tc_mode(e) && e->fuse_gather;
    int rc = run_network(e, n, st, fused ? &g : nullptr);
    e->d_value = saved;
    SCB_CHECK(rc);
    if (!fused) {
        SCB_CHECK(launch_policy_gather(e->logits, g.pos, g.moves, g.off, nullptr, n, g.priors, st));
        e->launches += 1;
    }
    return finish_timing(e, st);
}

int sc_eval(sc_engine *e, int n, const sc_position *pos, const sc_move *moves, const int32_t *move_off,
            float *priors_out, float *value_out, void *stream)
{
    SCB_CHECK(check_owner(e, "sc_eval"));
    if (!e || n < 0 || n > e->max_batch || (n > 0 && (!pos || !moves || !move_off || !priors_out || !value_out))) {
        set_error("sc_eval: bad argument");
        return SC_E_INVAL;
    }
    if (n == 0) return SC_OK;
    NvtxRange nv_call("sc_eval");
    const int total = move_off[n];
    bool mono = move_off[0] == 0 && total >= 0 && total <= e->max_moves_total;
    for (int i = 0; mono && i < n; i++) mono = move_off[i + 1] >= move_off[i];
    if (!mono) {
        set_error("sc_eval: bad move offsets");
        return SC_E_INVAL;
    }
    cudaStream_t st = stream ? (cudaStream_t)stream : e->stream;
    SCB_CUDA(cudaSetDevice(e->device));
    if (n <= SC_SMALL_N && total <= n * SC_MAX_MOVES) {  // (the staging buffers hold SC_MAX_MOVES moves per leaf)
        // latency path: [positions | offsets | moves] in one copy, [values | priors] back in one copy
        const size_t pos_b = sizeof(sc_position) * (size_t)n, off_b = sizeof(int32_t) * (size_t)(n + 1);
        const size_t mv_b = sizeof(sc_move) * (size_t)total;
        memcpy(e->h_small_in, pos, pos_b);
        memcpy(e->h_small_in + pos_b, move_off, off_b);
        memcpy(e->h_small_in + pos_b + off_b, moves, mv_b);
        // inputs: up to 16 leaves are read by the kernels straight from the pinned staging buffer (a few hundred bytes per
        // leaf over PCIe inside the encode / gather kernels instead of a copy engine round trip before the first launch)
        const uint8_t *in_dev = e->d_small_in;
        if (n <= 16)
            in_dev = e->h_small_in;
        else
            SCB_CUDA(cudaMemcpyAsync(e->d_small_in, e->h_small_in, pos_b + off_b + mv_b, cudaMemcpyHostToDevice, st));
        // results: the kernels store priors and values straight into the pinned (device-mapped under UVA) staging buffer --
        // posted writes over PCIe instead of a device buffer + a copy; the stream sync makes them visible to the host
        SCB_CHECK(sc_eval_device(e, n, in_dev, in_dev + pos_b + off_b, in_dev + pos_b, total, e->h_small_out + n, e->h_small_out, st));
        SCB_CUDA(cudaStreamSynchronize(st));
        memcpy(value_out, e->h_small_out, sizeof(float) * (size_t)n);
        memcpy(priors_out, e->h_small_out + n, sizeof(float) * (size_t)total);
        return SC_OK;
    }
    SCB_CUDA(cudaMemcpyAsync(e->d_pos, pos, sizeof(sc_position) * (size_t)n, cudaMemcpyHostToDevice, st));
    SCB_CUDA(cudaMemcpyAsync(e->d_off, move_off, sizeof(int32_t) * (size_t)(n + 1), cudaMemcpyHostToDevice, st));
    if (total) SCB_CUDA(cudaMemcpyAsync(e->d_moves, moves, sizeof(sc_move) * (size_t)total, cudaMemcpyHostToDevice, st));
    SCB_CHECK(sc_eval_device(e, n, e->d_pos, e->d_moves, e->d_off, total, e->d_priors, e->d_value, st));
    if (total) SCB_CUDA(cudaMemcpyAsync(priors_out, e->d_priors, sizeof(float) * (size_t)total, cudaMemcpyDeviceToHost, st));
    SCB_CUDA(cudaMemcpyAsync(value_out, e->d_value, sizeof(float) * (size_t)n, cudaMemcpyDeviceToHost, st));
    SCB_CUDA(cudaStreamSynchronize(st));
    return SC_OK;
}

int sc_predict(sc_engine *e, int n, const sc_position *pos, const int8_t *ep_square, sc_move *moves_out,
               int32_t *move_cnt_out, float *priors_out, float *value_out, void *stream)
{
    SCB_CHECK(check_owner(e, "sc_predict"));
    if (!e || n < 0 || n > e->max_batch ||
        (n > 0 && (!pos || !moves_out || !move_cnt_out || !priors_out || !value_out))) {
        set_error("sc_predict: bad argument");
        return SC_E_INVAL;
    }
    for (int i = 0; ep_square && i < n; i++) {
        const int s = ep_square[i];
        if (s != -1 && !(s >= 16 && s < 24) && !(s >= 40 && s < 48)) {
            set_error("sc_predict: ep_square[" + std::to_string(i) + "] = " + std::to_string(s) +
                      " is neither -1 nor a square of rank 3 or 6");
            return SC_E_INVAL;
        }
    }
    if (n == 0) return SC_OK;
    NvtxRange nv_call("sc_predict");
    cudaStream_t st = stream ? (cudaStream_t)stream : e->stream;
    SCB_CUDA(cudaSetDevice(e->device));
    SCB_CHECK(predict_setup(e));
    const size_t pos_b = sizeof(sc_position) * (size_t)n;
    const sc_position *d_pos;
    const int8_t *d_ep = nullptr;
    if (n <= SC_SMALL_N) {
        // sc_eval's staging: [positions | ep squares] in one pinned buffer, read in place by the kernels for up to 16
        // leaves, else one copy
        memcpy(e->h_small_in, pos, pos_b);
        if (ep_square) memcpy(e->h_small_in + pos_b, ep_square, (size_t)n);
        const uint8_t *in_dev = e->d_small_in;
        if (n <= 16)
            in_dev = e->h_small_in;
        else
            SCB_CUDA(cudaMemcpyAsync(e->d_small_in, e->h_small_in, pos_b + (ep_square ? n : 0), cudaMemcpyHostToDevice, st));
        d_pos = reinterpret_cast<const sc_position *>(in_dev);
        if (ep_square) d_ep = reinterpret_cast<const int8_t *>(in_dev + pos_b);
    } else {
        SCB_CUDA(cudaMemcpyAsync(e->d_pos, pos, pos_b, cudaMemcpyHostToDevice, st));
        if (ep_square) {
            SCB_CUDA(cudaMemcpyAsync(e->d_pred_ep, ep_square, (size_t)n, cudaMemcpyHostToDevice, st));
            d_ep = e->d_pred_ep;
        }
        d_pos = e->d_pos;
    }
    SCB_CHECK(predict_launch(e, n, d_pos, d_ep, priors_out, value_out, st));
    return predict_collect(e, "sc_predict", n, moves_out, move_cnt_out, priors_out, value_out, st,
                           [pos](int i) { return pos[i].meta[0] != 0; });
}

int sc_predict_stack(sc_engine *e, int n, const sc_move *stack, const int32_t *stack_off, const int8_t *n_hist,
                     sc_position *pos_out, sc_move *moves_out, int32_t *move_cnt_out, float *priors_out,
                     float *value_out, void *stream)
{
    SCB_CHECK(check_owner(e, "sc_predict_stack"));
    if (!e || n < 0 || n > e->max_batch ||
        (n > 0 && (!stack_off || !moves_out || !move_cnt_out || !priors_out || !value_out))) {
        set_error("sc_predict_stack: bad argument");
        return SC_E_INVAL;
    }
    if (n == 0) return SC_OK;
    NvtxRange nv_call("sc_predict_stack");
    return predict_replay(e, "sc_predict_stack", n, nullptr, nullptr, stack, stack_off, "stack_off", "stack", n_hist, pos_out,
                          moves_out, move_cnt_out, priors_out, value_out, &e->last_replay_ms, stream);
}

int sc_set_roots(sc_engine *e, int n_roots, const sc_move *stack, const int32_t *stack_off)
{
    SCB_CHECK(check_owner(e, "sc_set_roots"));
    if (!e || n_roots < 0 || n_roots > e->max_batch || (n_roots > 0 && !stack_off)) {
        set_error("sc_set_roots: bad argument");
        return SC_E_INVAL;
    }
    if (n_roots > 0)
        SCB_CHECK(check_move_lists("sc_set_roots", "root", "stack_off", "stack", n_roots, stack, stack_off, nullptr,
                                   [](int) { return 0; }));
    NvtxRange nv_call("sc_set_roots");
    e->n_roots = 0;
    if (n_roots == 0) return SC_OK;
    cudaStream_t st = e->stream;
    SCB_CUDA(cudaSetDevice(e->device));
    const int total = stack_off[n_roots];
    SCB_CHECK(roots_setup(e, (int64_t)total + n_roots));
    // the offsets stay on the device with the table: sc_predict_path finds each root's records through them
    SCB_CUDA(cudaMemcpyAsync(e->d_root_off, stack_off, sizeof(int32_t) * ((size_t)n_roots + 1), cudaMemcpyHostToDevice, st));
    if (total) SCB_CUDA(cudaMemcpyAsync(e->d_stack, stack, sizeof(sc_move) * (size_t)total, cudaMemcpyHostToDevice, st));
    SCB_CHECK(launch_root_replay(e->d_stack, e->d_root_off, n_roots, e->d_root_rec, e->d_root_pos, e->d_replay_status, st));
    e->launches += 1;
    SCB_CUDA(cudaMemcpyAsync(e->h_replay_status, e->d_replay_status, sizeof(int32_t) * (size_t)n_roots,
                             cudaMemcpyDeviceToHost, st));
    SCB_CUDA(cudaStreamSynchronize(st));
    for (int r = 0; r < n_roots; r++) {
        const int32_t status = e->h_replay_status[r];
        if (!status) continue;
        set_error(replay_error("sc_set_roots", "root", r, status >> 3, status));
        return SC_E_INVAL;
    }
    e->root_off.assign(stack_off, stack_off + n_roots + 1);
    e->n_roots = n_roots;
    return SC_OK;
}

int sc_predict_path(sc_engine *e, int n, const int32_t *root, const sc_move *path, const int32_t *path_off,
                    const int8_t *n_hist, sc_position *pos_out, sc_move *moves_out, int32_t *move_cnt_out,
                    float *priors_out, float *value_out, void *stream)
{
    SCB_CHECK(check_owner(e, "sc_predict_path"));
    if (!e || n < 0 || n > e->max_batch ||
        (n > 0 && (!root || !path_off || !moves_out || !move_cnt_out || !priors_out || !value_out))) {
        set_error("sc_predict_path: bad argument");
        return SC_E_INVAL;
    }
    if (e->n_roots == 0) {
        set_error("sc_predict_path: no roots are set (sc_set_roots)");
        return SC_E_STATE;
    }
    if (n == 0) return SC_OK;
    for (int i = 0; i < n; i++) {
        if (root[i] < 0 || root[i] >= e->n_roots) {
            set_error("sc_predict_path: root[" + std::to_string(i) + "] = " + std::to_string(root[i]) + " is not in 0.." +
                      std::to_string(e->n_roots - 1));
            return SC_E_INVAL;
        }
    }
    NvtxRange nv_call("sc_predict_path");
    return predict_replay(e, "sc_predict_path", n, root, nullptr, path, path_off, "path_off", "path", n_hist, pos_out,
                          moves_out, move_cnt_out, priors_out, value_out, &e->last_path_ms, stream);
}

int sc_eval_submit(sc_engine *e, int n, const sc_position *pos, const sc_move *moves_strided, const int32_t *move_cnt,
                   float *priors_out_strided, float *value_out, void *stream, int *ticket)
{
    SCB_CHECK(check_owner(e, "sc_eval_submit"));
    if (!e || !ticket || n < 0 || n > e->max_batch ||
        (n > 0 && (!pos || !moves_strided || !move_cnt || !priors_out_strided || !value_out))) {
        set_error("sc_eval_submit: bad argument");
        return SC_E_INVAL;
    }
    NvtxRange nv_call("sc_eval_submit");
    cudaStream_t st = stream ? (cudaStream_t)stream : e->stream;
    SCB_CUDA(cudaSetDevice(e->device));
    const int t = e->next_ticket;
    e->next_ticket = (t + 1) % SC_MAX_INFLIGHT;
    if (!e->tickets[t]) SCB_CUDA(cudaEventCreateWithFlags(&e->tickets[t], cudaEventDisableTiming));
    if (!e->copy_in) {
        SCB_CUDA(cudaStreamCreateWithFlags(&e->copy_in, cudaStreamNonBlocking));
        SCB_CUDA(cudaStreamCreateWithFlags(&e->copy_out, cudaStreamNonBlocking));
        for (auto &s : e->io) {
            SCB_CHECK(dev_alloc(e, &s.pos, (size_t)e->max_batch));
            SCB_CHECK(dev_alloc(e, &s.moves, (size_t)e->max_batch * SC_MAX_MOVES));
            SCB_CHECK(dev_alloc(e, &s.cnt, (size_t)e->max_batch));
            SCB_CHECK(dev_alloc(e, &s.priors, (size_t)e->max_batch * SC_MAX_MOVES));
            SCB_CHECK(dev_alloc(e, &s.value, (size_t)e->max_batch));
            SCB_CUDA(cudaEventCreateWithFlags(&s.in_done, cudaEventDisableTiming));
            SCB_CUDA(cudaEventCreateWithFlags(&s.compute_done, cudaEventDisableTiming));
            SCB_CUDA(cudaEventCreateWithFlags(&s.out_done, cudaEventDisableTiming));
        }
    }
    sc_engine::IoSet &io = e->io[e->n_submits & 1];
    const bool reused = e->n_submits >= 2;
    e->n_submits++;
    if (n > 0) {
        // inputs: wait until the kernels of the batch that used this set two submits ago are done with them
        if (reused) SCB_CUDA(cudaStreamWaitEvent(e->copy_in, io.compute_done, 0));
        SCB_CUDA(cudaMemcpyAsync(io.pos, pos, sizeof(sc_position) * (size_t)n, cudaMemcpyHostToDevice, e->copy_in));
        SCB_CUDA(cudaMemcpyAsync(io.cnt, move_cnt, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, e->copy_in));
        // strided by SC_MAX_MOVES on both sides, but only the first max(move_cnt) moves of every leaf travel
        int wmax = 1;
        for (int i = 0; i < n; i++) wmax = move_cnt[i] > wmax ? move_cnt[i] : wmax;
        if (wmax > SC_MAX_MOVES) wmax = SC_MAX_MOVES;
        SCB_CUDA(cudaMemcpy2DAsync(io.moves, sizeof(sc_move) * SC_MAX_MOVES, moves_strided, sizeof(sc_move) * SC_MAX_MOVES,
                                   sizeof(sc_move) * (size_t)wmax, (size_t)n, cudaMemcpyHostToDevice, e->copy_in));
        SCB_CUDA(cudaEventRecord(io.in_done, e->copy_in));
        // kernels: after the inputs arrived and after the previous results of this set left the device
        SCB_CUDA(cudaStreamWaitEvent(st, io.in_done, 0));
        if (reused) SCB_CUDA(cudaStreamWaitEvent(st, io.out_done, 0));
        SCB_CHECK(encode_for_mode(e, io.pos, n, st));
        const int saved_timing = e->timing;
        e->timing = 0;  // asynchronous path never synchronises
        const TcGather g{io.pos, io.moves, nullptr, io.cnt, io.priors, n};
        const bool fused = tc_mode(e) && e->fuse_gather;
        float *saved_value = e->d_value;
        e->d_value = io.value;
        int rc = run_network(e, n, st, fused ? &g : nullptr);
        e->d_value = saved_value;
        e->timing = saved_timing;
        SCB_CHECK(rc);
        if (!fused) {
            SCB_CHECK(launch_policy_gather(e->logits, g.pos, g.moves, nullptr, g.cnt, n, g.priors, st));
            e->launches += 1;
        }
        SCB_CUDA(cudaEventRecord(io.compute_done, st));
        // results
        SCB_CUDA(cudaStreamWaitEvent(e->copy_out, io.compute_done, 0));
        SCB_CUDA(cudaMemcpy2DAsync(priors_out_strided, sizeof(float) * SC_MAX_MOVES, io.priors, sizeof(float) * SC_MAX_MOVES,
                                   sizeof(float) * (size_t)wmax, (size_t)n, cudaMemcpyDeviceToHost, e->copy_out));
        SCB_CUDA(cudaMemcpyAsync(value_out, io.value, sizeof(float) * (size_t)n, cudaMemcpyDeviceToHost, e->copy_out));
        SCB_CUDA(cudaEventRecord(io.out_done, e->copy_out));
        SCB_CUDA(cudaEventRecord(e->tickets[t], e->copy_out));
    } else {
        SCB_CUDA(cudaEventRecord(io.in_done, e->copy_in));
        SCB_CUDA(cudaEventRecord(io.compute_done, st));
        SCB_CUDA(cudaEventRecord(io.out_done, e->copy_out));
        SCB_CUDA(cudaEventRecord(e->tickets[t], st));
    }
    *ticket = t;
    return SC_OK;
}

int sc_eval_wait(sc_engine *e, int ticket)
{
    SCB_CHECK(check_owner(e, "sc_eval_wait"));
    if (!e || ticket < 0 || ticket >= SC_MAX_INFLIGHT || !e->tickets[ticket]) {
        set_error("sc_eval_wait: bad ticket");
        return SC_E_INVAL;
    }
    NvtxRange nv_call("sc_eval_wait");
    SCB_CUDA(cudaEventSynchronize(e->tickets[ticket]));
    return SC_OK;
}

int sc_encode_only(sc_engine *e, int n, const sc_position *pos, int8_t *planes_out, int32_t *meta_out)
{
    SCB_CHECK(check_owner(e, "sc_encode_only"));
    if (!e || n < 0 || n > e->max_batch || (n > 0 && (!pos || !planes_out || !meta_out))) {
        set_error("sc_encode_only: bad argument");
        return SC_E_INVAL;
    }
    if (n == 0) return SC_OK;
    cudaStream_t st = e->stream;
    SCB_CUDA(cudaSetDevice(e->device));
    int8_t *d_planes = static_cast<int8_t *>(e->d_scratch);
    int32_t *d_meta = reinterpret_cast<int32_t *>(d_planes + (((size_t)n * 64 * SC_N_PLANES + 255) & ~(size_t)255));
    SCB_CUDA(cudaMemcpyAsync(e->d_pos, pos, sizeof(sc_position) * (size_t)n, cudaMemcpyHostToDevice, st));
    SCB_CHECK(launch_encode_i8(e->d_pos, n, d_planes, d_meta, st));
    e->launches += 1;
    SCB_CUDA(cudaMemcpyAsync(planes_out, d_planes, (size_t)n * 64 * SC_N_PLANES, cudaMemcpyDeviceToHost, st));
    SCB_CUDA(cudaMemcpyAsync(meta_out, d_meta, (size_t)n * SC_N_META * 4, cudaMemcpyDeviceToHost, st));
    SCB_CUDA(cudaStreamSynchronize(st));
    return SC_OK;
}

int sc_move_index_only(sc_engine *e, int n, const sc_position *pos, const sc_move *moves, const int32_t *move_off,
                       int32_t *index_out)
{
    SCB_CHECK(check_owner(e, "sc_move_index_only"));
    if (!e || n < 0 || n > e->max_batch || (n > 0 && (!pos || !moves || !move_off || !index_out))) {
        set_error("sc_move_index_only: bad argument");
        return SC_E_INVAL;
    }
    if (n == 0) return SC_OK;
    const int total = move_off[n];
    if (total < 0 || total > e->max_moves_total) {
        set_error("sc_move_index_only: bad move offsets");
        return SC_E_INVAL;
    }
    if (total == 0) return SC_OK;
    cudaStream_t st = e->stream;
    SCB_CUDA(cudaSetDevice(e->device));
    SCB_CUDA(cudaMemcpyAsync(e->d_pos, pos, sizeof(sc_position) * (size_t)n, cudaMemcpyHostToDevice, st));
    SCB_CUDA(cudaMemcpyAsync(e->d_off, move_off, sizeof(int32_t) * (size_t)(n + 1), cudaMemcpyHostToDevice, st));
    SCB_CUDA(cudaMemcpyAsync(e->d_moves, moves, sizeof(sc_move) * (size_t)total, cudaMemcpyHostToDevice, st));
    SCB_CHECK(launch_move_index(e->d_pos, e->d_moves, e->d_off, n, e->d_index, st));
    e->launches += 1;
    SCB_CUDA(cudaMemcpyAsync(index_out, e->d_index, sizeof(int32_t) * (size_t)total, cudaMemcpyDeviceToHost, st));
    SCB_CUDA(cudaStreamSynchronize(st));
    return SC_OK;
}

int sc_encode_steps(sc_engine *e, int n, const sc_move *played, const sc_move *child_moves,
                    const uint32_t *child_counts, const int32_t *child_off, int apply_mirror, int8_t *planes_out,
                    int32_t *meta_out, float *dist_out, int32_t *index_out, int32_t *index_off)
{
    SCB_CHECK(check_owner(e, "sc_encode_steps"));
    if (!e || n < 0 || n > e->max_batch ||
        (n > 0 && (!played || !child_moves || !child_counts || !child_off || !planes_out || !meta_out || !dist_out ||
                   !index_out || !index_off))) {
        set_error("sc_encode_steps: bad argument");
        return SC_E_INVAL;
    }
    if (n == 0) return SC_OK;
    if (child_off[0] != 0) {
        set_error("sc_encode_steps: child_off[0] must be 0");
        return SC_E_INVAL;
    }
    for (int i = 0; i < n; i++)
        if (child_off[i + 1] < child_off[i]) {
            set_error("sc_encode_steps: child_off must be non-decreasing");
            return SC_E_INVAL;
        }
    // ---- host: replay with the native rules (the reference replays through python-chess) -------------
    chess::Game g;
    std::vector<sc_position> pos((size_t)n);
    std::vector<sc_move> legal;
    std::vector<int32_t> loff((size_t)n + 1, 0);
    for (int i = 0; i < n; i++) {
        chess::MoveList l;
        g.cur.legal_moves(l);
        // the reference compares the SET of children with the SET of legal moves (src/lib.rs:84-96): every legal
        // move must be hit exactly once, so a duplicated child cannot stand in for a missing one
        const int cb = child_off[i], ce = child_off[i + 1];
        bool ok = (ce - cb) == l.n;
        bool seen[256] = {false};
        for (int k = cb; ok && k < ce; k++) {
            int hit = -1;
            for (int j = 0; j < l.n && hit < 0; j++)
                if (l.m[j].from == child_moves[k].from && l.m[j].to == child_moves[k].to &&
                    l.m[j].promo == child_moves[k].promo)
                    hit = j;
            ok = hit >= 0 && !seen[hit];
            if (ok) seen[hit] = true;
        }
        if (!ok) {
            set_error("sc_encode_steps: inconsistent moves at ply " + std::to_string(i));
            return SC_E_INVAL;
        }
        chess::Move mv{played[i].from, played[i].to, played[i].promo};
        bool in = false;
        for (int j = 0; j < l.n; j++) in = in || (l.m[j] == mv);
        if (!in) {
            set_error("sc_encode_steps: num_act table doesn't include the next move at ply " + std::to_string(i));
            return SC_E_INVAL;
        }
        // the packed leaf of ply i: full history back to the start (BoardHistory of lib.rs:52, capacity 8)
        host::pack_position(g, SC_LOOKBACK, &pos[i]);
        for (int j = 0; j < l.n; j++) legal.push_back(sc_move{l.m[j].from, l.m[j].to, l.m[j].promo, 0});
        loff[i + 1] = (int32_t)legal.size();
        g.push(mv);
    }
    const int n_child = child_off[n], n_legal = loff[n];
    if (n_child > e->max_moves_total || n_legal > e->max_moves_total) {
        set_error("sc_encode_steps: too many moves");
        return SC_E_INVAL;
    }
    // ---- device: planes, move indices of the legal moves, scattered visit distribution ---------------
    cudaStream_t st = e->stream;
    SCB_CUDA(cudaSetDevice(e->device));
    int8_t *d_planes = static_cast<int8_t *>(e->d_scratch);
    const size_t planes_bytes = ((size_t)n * 64 * SC_N_PLANES + 255) & ~(size_t)255;
    int32_t *d_meta = reinterpret_cast<int32_t *>(d_planes + planes_bytes);
    float *d_dist = reinterpret_cast<float *>(d_planes + planes_bytes + (((size_t)n * SC_N_META * 4 + 255) & ~(size_t)255));
    uint32_t *d_counts = reinterpret_cast<uint32_t *>(e->d_priors);  // reuse: same element size and capacity
    SCB_CUDA(cudaMemcpyAsync(e->d_pos, pos.data(), sizeof(sc_position) * (size_t)n, cudaMemcpyHostToDevice, st));
    SCB_CHECK(launch_encode_i8(e->d_pos, n, d_planes, d_meta, st));
    SCB_CUDA(cudaMemcpyAsync(e->d_moves, legal.data(), sizeof(sc_move) * (size_t)n_legal, cudaMemcpyHostToDevice, st));
    SCB_CUDA(cudaMemcpyAsync(e->d_off, loff.data(), sizeof(int32_t) * (size_t)(n + 1), cudaMemcpyHostToDevice, st));
    SCB_CHECK(launch_move_index(e->d_pos, e->d_moves, e->d_off, n, e->d_index, st));
    SCB_CUDA(cudaMemcpyAsync(index_out, e->d_index, sizeof(int32_t) * (size_t)n_legal, cudaMemcpyDeviceToHost, st));
    // children (trace order) -> dist
    SCB_CUDA(cudaMemcpyAsync(e->d_moves, child_moves, sizeof(sc_move) * (size_t)n_child, cudaMemcpyHostToDevice, st));
    SCB_CUDA(cudaMemcpyAsync(e->d_off, child_off, sizeof(int32_t) * (size_t)(n + 1), cudaMemcpyHostToDevice, st));
    SCB_CUDA(cudaMemcpyAsync(d_counts, child_counts, sizeof(uint32_t) * (size_t)n_child, cudaMemcpyHostToDevice, st));
    SCB_CHECK(launch_dist_scatter(e->d_pos, e->d_moves, d_counts, e->d_off, n, d_dist, st));
    e->launches += 3;
    SCB_CUDA(cudaMemcpyAsync(planes_out, d_planes, (size_t)n * 64 * SC_N_PLANES, cudaMemcpyDeviceToHost, st));
    SCB_CUDA(cudaMemcpyAsync(meta_out, d_meta, (size_t)n * SC_N_META * 4, cudaMemcpyDeviceToHost, st));
    SCB_CUDA(cudaMemcpyAsync(dist_out, d_dist, (size_t)n * SC_N_POLICY * 4, cudaMemcpyDeviceToHost, st));
    SCB_CUDA(cudaStreamSynchronize(st));
    memcpy(index_off, loff.data(), sizeof(int32_t) * (size_t)(n + 1));
    if (apply_mirror) {
        // `board_state.to_board().rotate()` (src/chess.rs:594-621) changes the meta, not the planes
        for (int i = 0; i < n; i++) {
            int32_t *m = meta_out + (size_t)i * SC_N_META;
            const int32_t t = m[0], k0 = m[2], q0 = m[3];
            m[1] += t == 1 ? 1 : 0;
            m[0] = !t;
            m[2] = m[4];
            m[3] = m[5];
            m[4] = k0;
            m[5] = q0;
        }
    }
    return SC_OK;
}

int sc_forward_only(sc_engine *e, int n, const float *planes, const float *meta, float *logp_out, float *value_out)
{
    SCB_CHECK(check_owner(e, "sc_forward_only"));
    if (!e || n < 0 || n > e->max_batch || (n > 0 && (!planes || !meta || !logp_out || !value_out))) {
        set_error("sc_forward_only: bad argument");
        return SC_E_INVAL;
    }
    if (n == 0) return SC_OK;
    cudaStream_t st = e->stream;
    SCB_CUDA(cudaSetDevice(e->device));
    float *d_nchw = static_cast<float *>(e->d_scratch);
    float *d_logp = d_nchw + (size_t)n * SC_N_PLANES * 64;
    SCB_CUDA(cudaMemcpyAsync(d_nchw, planes, (size_t)n * SC_N_PLANES * 64 * 4, cudaMemcpyHostToDevice, st));
    // meta rows are padded to 8 floats on the device
    SCB_CUDA(cudaMemsetAsync(e->d_meta, 0, (size_t)n * 8 * 4, st));
    SCB_CUDA(cudaMemcpy2DAsync(e->d_meta, 8 * 4, meta, SC_N_META * 4, SC_N_META * 4, (size_t)n, cudaMemcpyHostToDevice, st));
    if (e->mode == SC_MODE_FP32 && !e->fp32_tc)
        SCB_CHECK(launch_nchw_to_nhwc_f32(d_nchw, n, e->f_planes, st));
    else if (e->op == TC_OP_FP16)
        SCB_CHECK(launch_nchw_to_nhwc_fp16(d_nchw, n, reinterpret_cast<__half *>(e->h_planes), st));
    else if (e->op == TC_OP_E4M3)
        SCB_CHECK(launch_nchw_to_nhwc_e4m3(d_nchw, n, reinterpret_cast<uint8_t *>(e->h_planes), st));
    else
        SCB_CHECK(launch_nchw_to_nhwc_bf16(d_nchw, n, e->h_planes, st));
    e->launches += 1;
    if (e->timing) SCB_CUDA(cudaEventRecord(e->ev[0], st));
    SCB_CHECK(run_network(e, n, st));
    SCB_CHECK(launch_policy_logp_full(e->logits, n, d_logp, st));
    e->launches += 1;
    SCB_CHECK(finish_timing(e, st));
    SCB_CUDA(cudaMemcpyAsync(logp_out, d_logp, (size_t)n * SC_N_POLICY * 4, cudaMemcpyDeviceToHost, st));
    SCB_CUDA(cudaMemcpyAsync(value_out, e->d_value, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    SCB_CUDA(cudaStreamSynchronize(st));
    return SC_OK;
}

int sc_debug_tower(sc_engine *e, int n, const sc_position *pos, int n_layers, int which, uint16_t *x_out, uint16_t *t_out,
                   uint16_t *y_out)
{
    SCB_CHECK(check_owner(e, "sc_debug_tower"));
    if (!e || !tc_mode(e) || n <= 0 || n > e->max_batch || !pos || !e->tower) {
        set_error("sc_debug_tower: bad argument (bf16 / fp16 / fp8 engines only)");
        return SC_E_INVAL;
    }
    cudaStream_t st = e->stream;
    SCB_CUDA(cudaSetDevice(e->device));
    const size_t act = (size_t)e->alloc_boards * 64 * C_TOWER * 2;
    SCB_CUDA(cudaMemsetAsync(e->h_x, 0, act, st));
    SCB_CUDA(cudaMemsetAsync(e->h_t, 0, act, st));
    SCB_CUDA(cudaMemsetAsync(e->h_y, 0, act, st));
    SCB_CUDA(cudaMemcpyAsync(e->d_pos, pos, sizeof(sc_position) * (size_t)n, cudaMemcpyHostToDevice, st));
    SCB_CHECK(encode_for_mode(e, e->d_pos, n, st));
    if (which == 1) {
        if (!e->lat) {
            set_error("sc_debug_tower: no latency kernel");
            return SC_E_STATE;
        }
        int rc = lat_tower_launch(e->lat, n, st, n_layers);
        if (rc == SC_E_STATE) set_error("sc_debug_tower: batch too large for the latency kernel");
        SCB_CHECK(rc);
    } else
        SCB_CHECK(tc_tower_launch(e->tower, n, e->num_sms, e->tower_group, st, n_layers));
    const size_t count = (size_t)n * 64 * C_TOWER;
    if (e->op == TC_OP_E4M3) {
        // e4m3 bytes, widened to the fp16 bit patterns of the same values (exact)
        std::vector<uint8_t> h(count);
        const std::pair<uint16_t *, const void *> bufs[3] = {{x_out, e->h_x}, {t_out, e->h_t}, {y_out, e->h_y}};
        for (const auto &b : bufs) {
            if (!b.first) continue;
            SCB_CUDA(cudaMemcpyAsync(h.data(), b.second, count, cudaMemcpyDeviceToHost, st));
            SCB_CUDA(cudaStreamSynchronize(st));
            for (size_t i = 0; i < count; i++) b.first[i] = __nv_cvt_fp8_to_halfraw((__nv_fp8_storage_t)h[i], __NV_E4M3).x;
        }
        return SC_OK;
    }
    const size_t bytes = count * 2;
    if (x_out) SCB_CUDA(cudaMemcpyAsync(x_out, e->h_x, bytes, cudaMemcpyDeviceToHost, st));
    if (t_out) SCB_CUDA(cudaMemcpyAsync(t_out, e->h_t, bytes, cudaMemcpyDeviceToHost, st));
    if (y_out) SCB_CUDA(cudaMemcpyAsync(y_out, e->h_y, bytes, cudaMemcpyDeviceToHost, st));
    SCB_CUDA(cudaStreamSynchronize(st));
    return SC_OK;
}

int64_t sc_launch_count(const sc_engine *e) { return e ? e->launches : 0; }

int sc_set_timing(sc_engine *e, int enabled)
{
    SCB_CHECK(check_owner(e, "sc_set_timing"));
    if (!e) return SC_E_INVAL;
    e->timing = enabled < 0 ? 0 : (enabled > 2 ? 2 : enabled);
    return SC_OK;
}

double sc_timed_flops_per_leaf(const sc_engine *e) { return e ? e->timed_flops_per_leaf : 0.0; }

int sc_kernel_timing(sc_engine *e, float *conv3x3_avg_ms, int *n_launches)
{
    if (!e) return SC_E_INVAL;
    if (conv3x3_avg_ms) *conv3x3_avg_ms = e->last_conv_avg_ms;
    if (n_launches) *n_launches = e->last_conv_n;
    return SC_OK;
}

int sc_predict_timing(sc_engine *e, float *movegen_ms)
{
    if (!e) return SC_E_INVAL;
    if (movegen_ms) *movegen_ms = e->last_movegen_ms;
    return SC_OK;
}

int sc_predict_stack_timing(sc_engine *e, float *replay_ms)
{
    if (!e) return SC_E_INVAL;
    if (replay_ms) *replay_ms = e->last_replay_ms;
    return SC_OK;
}

int sc_predict_path_timing(sc_engine *e, float *replay_ms)
{
    if (!e) return SC_E_INVAL;
    if (replay_ms) *replay_ms = e->last_path_ms;
    return SC_OK;
}

int sc_last_timing(sc_engine *e, float *tower_ms, float *total_ms)
{
    if (!e) return SC_E_INVAL;
    if (tower_ms) *tower_ms = e->last_tower_ms;
    if (total_ms) *total_ms = e->last_total_ms;
    return SC_OK;
}

}  // extern "C"
