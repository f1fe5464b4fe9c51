// Latency path of the bf16 network for small batches (the `Game::predict` drop-in, src/backends/torch.rs:115-125, is a
// batch of ONE): the same arithmetic as tower_bf16.cu, bit for bit, laid out for latency instead of throughput.
//
// tower_bf16.cu gives a 4-board tile to one CTA pair and walks the 41 convolutions with it: for a batch of <= 4 boards
// two SMs work and 146 idle (~18 us per layer, 0.75 ms per call).  Here a tile is TWO boards (128 rows) and its 256
// output channels are split over a thread-block cluster of CL = 8 (32 channels per CTA) or 4 (64 per CTA) CTAs, all
// layers in one launch:
//   * every CTA loads the tile's full activations (A, TMA box {64 ch, 8 files, 2 boards, 10 ranks} per (channel chunk,
//     dx), three dy taps per box as in tower_bf16.cu) and ITS slice of the weights (B, box {64, NC, 1, 3}: the three dy
//     taps of (chunk, dx) in one load) and issues tcgen05.mma M128 x N(NC) x K16 in the throughput kernel's k order;
//   * LayerNorm needs statistics over all 256 channels of a row: every CTA pushes its per-32-channel partial sums into
//     the shared memory of all CTAs of the cluster (st.shared::cluster) and signals their mbarriers; the partials are
//     combined in the fixed tree of tc_ptx.cuh, which is what makes the result identical to the throughput kernel;
//   * squeeze-excitation: the channel means of a CTA's own channels stay local; FC1 is defined per 32-channel chunk
//     (tc_ptx.cuh), so every CTA computes ITS chunks' partial sums for all 128 hidden units and pushes them to the
//     cluster -- one exchange -- and everybody adds the eight partials in the fixed tree; FC2 and the gate are per
//     channel, i.e. local;
//   * layer l+1 reads layer l's output through L2: the epilogue threads put the CTA's slice into a shared-memory tile
//     laid out as the TMA box {NC channels, 8 files, boards, 8 ranks}, ONE thread stores it (cp.async.bulk.tensor) and
//     waits for the write to complete, then the CTA signals the `ready` mbarrier of every CTA of the cluster, whose TMA
//     warp starts the next layer's activation loads (128 threads storing to global memory and fencing generic -> async
//     proxy at GPU scope cost 0.9 k cycles per layer more).  Weight loads never wait for
//     activations: their producer warp runs ahead through the layers as far as its ring allows.
// A tile of ONE board (NB = 1: 64 rows, tcgen05.mma M64) halves the shared-memory operand traffic that bounds the MMA
// phase at these narrow N; it is used while there are enough clusters for one board each.
// (An epilogue of eight warps -- two per TMEM quadrant, half of the CTA's channels each -- was built and measured: the
// per-thread work halves, but twice as many threads fence and push statistics; 541 k cycles per call against 524 k.)
// Warp roles (256 threads): 0 = activation TMA, 1 = weight TMA, 2 = TMEM allocator + MMA issuer, 3 = SE weight
// staging, 4..7 = epilogue (one thread per row of the tile).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "common.cuh"
#include "tc_host.cuh"
#include "tc_ptx.cuh"

namespace scb {

constexpr int LAT_THREADS = 256;

struct alignas(64) LatLayer {
    CUtensorMap map_a;   // input activations {C, file, board, rank}, box of two boards
    CUtensorMap map_a1;  // the same tensor, box of one board
    CUtensorMap map_w;  // weights {cin, cout, dx, dy}, box {64, NC, 1, 3 | 1}
    CUtensorMap map_o, map_o1;  // output {C, file, board, rank}, box {NC, 8, 2 | 1, 8}, no swizzle (TMA store hand-over)
    const __nv_bfloat16 *resid;
    const float *bias, *gamma, *beta;
    const uint4 *se_w1s, *se_w2s;  // per cluster rank: fc1 columns [NC / 8][128] x 8 bf16, fc2 rows [16][NC] x 8 bf16
    const float *se_b1, *se_b2;
    int taps, kchunks, relu, se, ln;
};

struct LatArgs {
    const LatLayer *layers;
    int n_layers;
    int n_tiles;
    long long *prof;  // optional [grid][16] cycle counters (SCB200_PHASE_PROFILE=1)
};

template <int CL, int NB = 2> struct LatCfg {
    static constexpr int NC = 256 / CL;  // output channels per CTA
    static constexpr int HJ = 128 / CL;  // SE hidden units per CTA
    static constexpr int A_BOX = NB * 80 * TC_BK * 2;  // 10 ranks x NB boards x 8 files rows of 128 B
    static constexpr int B_TILE = 3 * NC * TC_BK * 2;
    // one pipeline stage = the activation box and the weight tile of a (channel chunk, dx) step; both loads complete on
    // the stage's one `full` barrier (a wait on an already complete mbarrier still costs ~90 cycles, and a layer has
    // only 12 steps), but they are issued by two warps so that the weights can run ahead of the activations
    static constexpr int STAGE = A_BOX + B_TILE;
    static constexpr int NS = (160 * 1024) / STAGE;
    static constexpr int W1S_BYTES = 32 * HJ * 16, W2S_BYTES = 16 * NC * 16;
    static constexpr int OFF_W1S = NS * STAGE;
    static constexpr int OFF_W2S = OFF_W1S + W1S_BYTES;
    static constexpr int OFF_STAT = OFF_W2S + W2S_BYTES;  // float2 [8 chunks][128 rows]
    static constexpr int OFF_PAR = OFF_STAT + 8 * 128 * 8;  // bias, gamma, beta [NC]
    static constexpr int OFF_POOL = OFF_PAR + 2 * 3 * NC * 4;  // (parameters double-buffered by layer parity) [4 quads][2 boards][NC]
    static constexpr int OFF_MEAN = OFF_POOL + 8 * NC * 4;   // [NB][NC] means of this CTA's channels
    static constexpr int OFF_HIDP = OFF_MEAN + 2 * NC * 4;   // [8 chunks][2 boards][128] FC1 chunk partials (pushed by the cluster)
    static constexpr int OFF_HID = OFF_HIDP + 8 * 2 * 128 * 4;  // [2][128]
    static constexpr int OFF_FC2P = OFF_HID + 2 * 128 * 4;      // [2 * NC outputs][4 chunk sums]
    static constexpr int OFF_GATE = OFF_FC2P + 2 * NC * 4 * 4;  // [2][NC]
    static constexpr int OFF_OUT = (OFF_GATE + 2 * NC * 4 + 127) & ~127;  // [64 NB rows][NC] bf16 output staging (TMA store)
    static constexpr int OFF_BARS = OFF_OUT + 128 * NC * 2;
    static constexpr int N_BARS = 2 * 8 + 7;  // up to 8 stages (full, empty) + 7 single barriers, the same in every variant
    static constexpr int SMEM_BYTES = OFF_BARS + N_BARS * 8 + 16;
};

__device__ __forceinline__ uint32_t map_to_cta(uint32_t addr, uint32_t cta)
{
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(cta));
    return r;
}
// store into the shared memory of a CTA of the cluster that also counts its bytes on an mbarrier of that CTA
// (st.async): the receiver waits for the byte count, no fence and no separate arrive on the sender's side
__device__ __forceinline__ void st_async_f32x2(uint32_t addr, float a, float b, uint32_t bar)
{
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f32 [%0], {%1, %2}, [%3];" ::"r"(addr),
                 "f"(a), "f"(b), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void st_async_f32(uint32_t addr, float a, uint32_t bar)
{
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.f32 [%0], %1, [%2];" ::"r"(addr), "f"(a),
                 "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr)
{
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity)
{
    uint32_t ok = 0;
    while (!ok) {
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}"
            : "=r"(ok)
            : "r"(bar), "r"(parity)
            : "memory");
    }
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
// Column sums over 16 lanes (lane bits 8, 4, 2, 1; bit 16 is not touched) of 32 per-lane values: the one-board tile's
// form of warp_transpose_reduce_2boards -- same tree (rank pair first, then files 4, 2, 1), so the same bits.  Lane l
// ends with the sums for indices i0, i0 + 1, i0 = 16 b8 + 8 b4 + 4 b2 + 2 b1.
__device__ __forceinline__ float2 warp_transpose_reduce_16(float (&v)[32], int lane, int &i0)
{
    const bool b8 = lane & 8, b4 = lane & 4, b2 = lane & 2, b1 = lane & 1;
    float w16[16], w8[8], w4[4], w2[2];
#pragma unroll
    for (int i = 0; i < 16; i++) {
        float send = b8 ? v[i] : v[i + 16];
        float keep = b8 ? v[i + 16] : v[i];
        w16[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
#pragma unroll
    for (int i = 0; i < 8; i++) {
        float send = b4 ? w16[i] : w16[i + 8];
        float keep = b4 ? w16[i + 8] : w16[i];
        w8[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
        float send = b2 ? w8[i] : w8[i + 4];
        float keep = b2 ? w8[i + 4] : w8[i];
        w4[i] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
    }
#pragma unroll
    for (int i = 0; i < 2; i++) {
        float send = b1 ? w4[i] : w4[i + 2];
        float keep = b1 ? w4[i + 2] : w4[i];
        w2[i] = keep + __shfl_xor_sync(0xffffffffu, send, 1);
    }
    i0 = (b8 ? 16 : 0) + (b4 ? 8 : 0) + (b2 ? 4 : 0) + (b1 ? 2 : 0);
    return make_float2(w2[0], w2[1]);
}

__device__ __forceinline__ void lat_epi_sync() { asm volatile("bar.sync 1, 128;" ::: "memory"); }


// OT: the operand type (OpBf16 / OpFp16, tc_ptx.cuh), the same as the throughput kernel's for the same engine
template <int CL, int NB, class OT = OpBf16>
__global__ void __launch_bounds__(LAT_THREADS, 1) lat_tower_kernel(const LatArgs args)
{
    using Cfg = LatCfg<CL, NB>;
    constexpr int A_BOX = Cfg::A_BOX, DY_STEP = NB * 1024;  // bytes between the dy taps inside an activation box
    constexpr int NC = Cfg::NC, NS = Cfg::NS;
    static_assert(NS >= 3 && NS <= 8, "stage count");
    constexpr int NCH = NC / 32;  // 32-channel chunks per CTA
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t smem_base = smem_u32(smem);
    if (smem_base & 1023u) __trap();
    float2 *s_stat = reinterpret_cast<float2 *>(smem + Cfg::OFF_STAT);
    float *s_par = reinterpret_cast<float *>(smem + Cfg::OFF_PAR);
    float *s_pool = reinterpret_cast<float *>(smem + Cfg::OFF_POOL);
    float *s_mean = reinterpret_cast<float *>(smem + Cfg::OFF_MEAN);
    float *s_hidp = reinterpret_cast<float *>(smem + Cfg::OFF_HIDP);
    float *s_hid = reinterpret_cast<float *>(smem + Cfg::OFF_HID);
    float *s_gate = reinterpret_cast<float *>(smem + Cfg::OFF_GATE);
    float *s_fc2p = reinterpret_cast<float *>(smem + Cfg::OFF_FC2P);
    const uint4 *s_w1s = reinterpret_cast<const uint4 *>(smem + Cfg::OFF_W1S);
    const uint4 *s_w2s = reinterpret_cast<const uint4 *>(smem + Cfg::OFF_W2S);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + Cfg::OFF_BARS);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + Cfg::N_BARS);
    const uint32_t bar_base = smem_u32(bars);
    auto full = [&](int s) { return bar_base + 8u * s; };
    auto empty = [&](int s) { return bar_base + 8u * (8 + s); };
    const uint32_t bar_tfull = bar_base + 8u * 16, bar_ready = bar_tfull + 8, bar_stat = bar_tfull + 16,
                   bar_mean = bar_tfull + 24, bar_hid = bar_tfull + 32, bar_sewf = bar_tfull + 40, bar_sewe = bar_tfull + 48;
    auto abox = [&](int s) { return smem_base + (uint32_t)(s * Cfg::STAGE); };
    auto btile = [&](int s) { return smem_base + (uint32_t)(s * Cfg::STAGE + A_BOX); };

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const uint32_t rank = __shfl_sync(0xffffffffu, cluster_ctarank(), 0);
    const int tile = (int)blockIdx.x / CL;
    const int n_layers = args.n_layers;

    if (threadIdx.x == 0) {
        for (int s = 0; s < 8; s++) {
            mbar_init(full(s), 2);   // the activation producer's and the weight producer's expect_tx arrivals
            mbar_init(empty(s), 1);  // the MMA warp's commit
        }
        mbar_init(bar_tfull, 1);
        mbar_init(bar_ready, CL);  // one arrival per CTA of the cluster
        mbar_init(bar_stat, 1);    // armed per layer with the bytes every CTA pushes (st.async)
        mbar_init(bar_mean, 1);
        mbar_init(bar_hid, 1);
        mbar_init(bar_sewf, 1);
        mbar_init(bar_sewe, 4);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"((uint32_t)(NC < 32 ? 32 : NC))
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();  // every CTA's barriers exist before any remote arrive
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) asm volatile("prefetch.tensormap [%0];" ::"l"(NB == 2 ? &args.layers[0].map_a : &args.layers[0].map_a1) : "memory");
        // ---- activation boxes: wait until the whole cluster has written the previous layer ----
        int st = 0;
        uint32_t ph = 0;
        long long pa_ready = 0, pa_empty = 0;
        for (int l = 0; l < n_layers; l++) {
            const LatLayer &L = args.layers[l];
            const int nd = L.taps == 9 ? 3 : 1;
            if (l > 0) {
                const long long t0 = args.prof ? clock64() : 0;
                mbar_wait_cluster(bar_ready, (uint32_t)(l - 1) & 1u);
                if (args.prof) pa_ready += clock64() - t0;
                // (no proxy fence on this side: the writers fenced generic -> async before they signalled, and the
                //  acquire above orders the TMA issue after the signal -- the same hand-over as tower_bf16.cu's)
            }
            for (int kc = 0; kc < L.kchunks; kc++)
                for (int dxi = 0; dxi < nd; dxi++) {
                    const long long t1 = args.prof ? clock64() : 0;
                    mbar_wait(empty(st), ph ^ 1u);
                    if (args.prof) pa_empty += clock64() - t1;
                    if (elect_one()) {
                        mbar_expect_tx(full(st), A_BOX);
                        tma_load_4d(abox(st), NB == 2 ? &L.map_a : &L.map_a1, full(st), kc * TC_BK, nd == 3 ? dxi - 1 : 0,
                                    tile * NB, -1);
                    }
                    __syncwarp();
                    if (++st == NS) {
                        st = 0;
                        ph ^= 1u;
                    }
                }
            // the next layer's tensor map (a different 128-byte descriptor per layer) would otherwise be fetched from
            // L2 on the critical path right after the hand-over
            if (l + 1 < n_layers && lane == 0)
                asm volatile("prefetch.tensormap [%0];" ::"l"(NB == 2 ? &args.layers[l + 1].map_a : &args.layers[l + 1].map_a1)
                             : "memory");
        }
        if (args.prof && lane == 0) {
            args.prof[blockIdx.x * 16 + 0] = pa_ready;
            args.prof[blockIdx.x * 16 + 1] = pa_empty;
        }
    } else if (warp == 1) {
        // ---- this CTA's slice of the weights; independent of the activations, runs ahead ----
        int st = 0;
        uint32_t ph = 0;
        for (int l = 0; l < n_layers; l++) {
            const LatLayer &L = args.layers[l];
            const int nd = L.taps == 9 ? 3 : 1;
            if (l + 1 < n_layers && lane == 0) asm volatile("prefetch.tensormap [%0];" ::"l"(&args.layers[l + 1].map_w) : "memory");
            for (int kc = 0; kc < L.kchunks; kc++)
                for (int dxi = 0; dxi < nd; dxi++) {
                    mbar_wait(empty(st), ph ^ 1u);
                    if (elect_one()) {
                        mbar_expect_tx(full(st), (uint32_t)(nd * NC * TC_BK * 2));
                        tma_load_4d(btile(st), &L.map_w, full(st), kc * TC_BK, (int)rank * NC, dxi, 0);
                    }
                    __syncwarp();
                    if (++st == NS) {
                        st = 0;
                        ph ^= 1u;
                    }
                }
        }
    } else if (warp == 2) {
        // ---- MMA issuer: k order (channel chunk, dx, dy, 16-element step) as in tower_bf16.cu ----
        constexpr uint32_t idesc = umma_idesc<OT>(64 * NB, NC);
        int rs = 0;
        uint32_t rph = 0;
        long long pm_a = 0, pm_a0 = 0, pm_total = args.prof ? clock64() : 0;
        for (int l = 0; l < n_layers; l++) {
            const LatLayer &L = args.layers[l];
            const int nd = L.taps == 9 ? 3 : 1;
            uint32_t acc = 0;
            for (int g = 0; g < L.kchunks * nd; g++) {
                const long long t0 = args.prof ? clock64() : 0;
                mbar_wait(full(rs), rph);
                if (args.prof) (g == 0 ? pm_a0 : pm_a) += clock64() - t0;
                tc_fence_after();
                const uint32_t a0 = abox(rs), b0 = btile(rs);
                if (elect_one()) {
                    for (int dyi = 0; dyi < nd; dyi++) {
                        const uint64_t da = umma_desc_sw128(a0 + (uint32_t)((nd == 3 ? dyi : 1) * DY_STEP));
                        const uint64_t db = umma_desc_sw128(b0 + (uint32_t)(dyi * NC * TC_BK * 2));
#pragma unroll
                        for (int k = 0; k < TC_BK / 16; k++)
                            tc_mma_bf16(tmem_base, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc,
                                        (acc | (uint32_t)dyi | (uint32_t)k) != 0);
                    }
                    tc_commit(empty(rs));
                }
                __syncwarp();
                acc = 1;
                if (++rs == NS) {
                    rs = 0;
                    rph ^= 1u;
                }
            }
            if (elect_one()) tc_commit(bar_tfull);
            __syncwarp();
        }
        if (args.prof && lane == 0) {
            args.prof[blockIdx.x * 16 + 2] = pm_a0;
            args.prof[blockIdx.x * 16 + 3] = pm_a;
            args.prof[blockIdx.x * 16 + 4] = 0;
            args.prof[blockIdx.x * 16 + 5] = clock64() - pm_total;
        }
    } else if (warp == 3) {
        // ---- SE weights of this CTA's hidden units (fc1) and channels (fc2) -> shared memory, one SE layer ahead ----
        int k = 0;
        for (int l = 0; l < n_layers; l++) {
            const LatLayer &L = args.layers[l];
            if (L.se != 1) continue;
            if (k > 0) mbar_wait(bar_sewe, (uint32_t)(k - 1) & 1u);  // the previous SE layer's FC2 has read them
            if (elect_one()) {
                mbar_expect_tx(bar_sewf, Cfg::W1S_BYTES + Cfg::W2S_BYTES);
                bulk_g2s(smem_base + Cfg::OFF_W1S, L.se_w1s + (size_t)rank * (Cfg::W1S_BYTES / 16), Cfg::W1S_BYTES, bar_sewf);
                bulk_g2s(smem_base + Cfg::OFF_W2S, L.se_w2s + (size_t)rank * (Cfg::W2S_BYTES / 16), Cfg::W2S_BYTES, bar_sewf);
            }
            __syncwarp();
            k++;
        }
    } else {
        // ---- epilogue.  NB = 2: thread = accumulator row (rank, board, file), TMEM lane = row.  NB = 1 (M64): the 64
        //      rows (rank, file) sit in lanes 0..15 of each 32-lane TMEM quadrant (row = 16 quad + lane); lanes 16..31
        //      carry nothing but take part in the warp-wide instructions. ----
        const int quad = warp & 3;
        const int tid = quad * 32 + lane;  // 0..127: index for the work that is not tied to a row
        const bool active = NB == 2 || lane < 16;
        const int row = NB == 2 ? tid : quad * 16 + (lane & 15);
        const int board = NB == 2 ? (row >> 3) & 1 : 0;
        const int orow = NB == 2 ? board * 64 + (row >> 4) * 8 + (row & 7) : row;  // the row's place in memory
        const int c0 = (int)rank * NC;
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16);
        const size_t grow = (size_t)tile * (64 * NB) + orow;
        int n_stat = 0, n_se = 0;
        const bool prof = args.prof != nullptr && tid == 0;
        long long pe_tfull = 0, pe_stat = 0, pe_se = 0, pe_work = 0, pe_ld = 0, pe_pfence = 0, pe_sync = 0, pe_gfence = 0;
        for (int l = 0; l < n_layers; l++) {
            const LatLayer &L = args.layers[l];
            // this layer's parameters; double-buffered, a slow warp may still be reading the previous layer's
            float *s_bias = s_par + (l & 1) * 3 * NC, *s_gamma = s_bias + NC, *s_beta = s_gamma + NC;
            if (tid < NC) {
                s_bias[tid] = L.bias[c0 + tid];
                s_gamma[tid] = L.ln ? L.gamma[c0 + tid] : 1.f;
                s_beta[tid] = L.ln ? L.beta[c0 + tid] : 0.f;
            }
            // the residual does not depend on this layer: request it before anything else
            uint4 xres[NC / 8];
            if (L.se && active) {
                const uint4 *xg = reinterpret_cast<const uint4 *>(L.resid + grow * 256 + c0);
#pragma unroll
                for (int i = 0; i < NC / 8; i++) xres[i] = xg[i];
            }
            // SE biases of this thread's hidden unit / channel: global loads, requested a whole MMA phase before their use
            float se_b1v = 0.f, se_b2v = 0.f;
            if (L.se == 1) {
                se_b1v = L.se_b1[tid];
                se_b2v = L.se_b2[c0 + tid % NC];
            }
            if (tid == 0) {
                // arm this layer's exchange barriers with the bytes the cluster will push into this CTA
                if (L.ln) mbar_expect_tx(bar_stat, 8 * 64 * NB * 8);
                if (L.se == 1) mbar_expect_tx(bar_hid, 8 * NB * 128 * 4);
            }
            lat_epi_sync();  // parameters visible
            const long long tp0 = prof ? clock64() : 0;
            mbar_wait(bar_tfull, (uint32_t)l & 1u);
            const long long tp1 = prof ? clock64() : 0;
            pe_tfull += tp1 - tp0;
            tc_fence_after();
            float a[NC];
#pragma unroll
            for (int ch = 0; ch < NCH; ch++) {
                uint32_t r[32];
                tmem_ld32(taddr + ch * 32, r);
#pragma unroll
                for (int j = 0; j < 32; j++) a[ch * 32 + j] = __fadd_rn(__uint_as_float(r[j]), s_bias[ch * 32 + j]);
            }
            tc_fence_before();
            if (prof) pe_ld += clock64() - tp1;
            float mean = 0.f, rstd = 1.f;
            if (L.ln) {
                // per-chunk partial sums -> every CTA of the cluster
                if (active) {
#pragma unroll
                    for (int ch = 0; ch < NCH; ch++) {
                        float av[32], sm, q;
#pragma unroll
                        for (int j = 0; j < 32; j++) av[j] = a[ch * 32 + j];
                        ln_chunk_stats(av, sm, q);
                        const uint32_t mine = smem_u32(s_stat + ((int)rank * NCH + ch) * 128 + row);
#pragma unroll
                        for (int c = 0; c < CL; c++)
                            st_async_f32x2(map_to_cta(mine, (uint32_t)c), sm, q, map_to_cta(bar_stat, (uint32_t)c));
                    }
                }
                const long long ts0 = prof ? clock64() : 0;
                mbar_wait_cluster(bar_stat, (uint32_t)n_stat & 1u);
                if (prof) pe_stat += clock64() - ts0;
                n_stat++;
                const float2 h0 = ln_half(s_stat[0 * 128 + row], s_stat[1 * 128 + row], s_stat[2 * 128 + row], s_stat[3 * 128 + row]);
                const float2 h1 = ln_half(s_stat[4 * 128 + row], s_stat[5 * 128 + row], s_stat[6 * 128 + row], s_stat[7 * 128 + row]);
                ln_finish(h0, h1, LN_EPS, mean, rstd);
            }
#pragma unroll
            for (int j = 0; j < NC; j++) a[j] = ln_apply(a[j], mean, rstd, s_gamma[j], s_beta[j]);
            // the row goes to the output staging tile [row][NC] (row = accumulator row = the store box's (rank, board, file)
            // order, so the tile is exactly the store box)
            uint4 *odst = reinterpret_cast<uint4 *>(smem + Cfg::OFF_OUT + row * NC * 2);
            if (!L.se) {
                // ---- bias + LayerNorm (+ReLU) -> operand type ----
                if (active) {
#pragma unroll
                    for (int i = 0; i < NC / 8; i++) {
                        uint32_t pw[4];
#pragma unroll
                        for (int k = 0; k < 4; k++) {
                            float y0 = a[8 * i + 2 * k], y1 = a[8 * i + 2 * k + 1];
                            if (L.relu) {
                                y0 = fmaxf(y0, 0.f);
                                y1 = fmaxf(y1, 0.f);
                            }
                            pw[k] = OT::pack2(y0, y1);
                        }
                        odst[i] = make_uint4(pw[0], pw[1], pw[2], pw[3]);
                    }
                }
            } else {
                const long long tq0 = prof ? clock64() : 0;
                if (L.se == 1) {
                    // ---- squeeze: channel sums of this warp's 16 rows per board, then over the four warps ----
#pragma unroll
                    for (int ch = 0; ch < NCH; ch++) {
                        float y[32];
#pragma unroll
                        for (int j = 0; j < 32; j++) y[j] = a[ch * 32 + j];
                        int i0;
                        const float2 ps = NB == 2 ? warp_transpose_reduce_2boards(y, lane, i0) : warp_transpose_reduce_16(y, lane, i0);
                        if (active) *reinterpret_cast<float2 *>(s_pool + (quad * NB + board) * NC + ch * 32 + i0) = ps;
                    }
                    lat_epi_sync();
                    if (tid < NB * NC) {
                        const int b = tid / NC, c = tid % NC;
                        s_mean[b * NC + c] = __fmul_rn(__fadd_rn(__fadd_rn(s_pool[b * NC + c], s_pool[(NB + b) * NC + c]),
                                                                 __fadd_rn(s_pool[(2 * NB + b) * NC + c], s_pool[(3 * NB + b) * NC + c])),
                                                       1.f / 64.f);
                    }
                    mbar_wait(bar_sewf, (uint32_t)n_se & 1u);  // this layer's SE weights are in shared memory
                    lat_epi_sync();
                    // ---- excitation FC1: thread = hidden unit; the chunk sums of THIS CTA's channels (one sequential fma
                    //      chain per chunk and board, as in tower_bf16.cu) go to every CTA of the cluster ----
                    {
                        const int j = tid;
#pragma unroll
                        for (int ch = 0; ch < NCH; ch++) {
                            float p0 = 0.f, p1 = 0.f;
#pragma unroll
                            for (int uu = 0; uu < 4; uu++) {
                                float wf[8];
                                OT::unpack8(s_w1s[(ch * 4 + uu) * 128 + j], wf);
                                const float *m = s_mean + ch * 32 + uu * 8;
                                p0 = se_chain8(wf, *reinterpret_cast<const float4 *>(m), *reinterpret_cast<const float4 *>(m + 4), p0);
                                if (NB == 2)
                                    p1 = se_chain8(wf, *reinterpret_cast<const float4 *>(m + NC),
                                                   *reinterpret_cast<const float4 *>(m + NC + 4), p1);
                            }
                            const int kg = (int)rank * NCH + ch;  // global chunk index 0..7
                            const uint32_t dst = smem_u32(s_hidp + (kg * 2 + 0) * 128 + j);
#pragma unroll
                            for (int cc = 0; cc < CL; cc++) {
                                st_async_f32(map_to_cta(dst, (uint32_t)cc), p0, map_to_cta(bar_hid, (uint32_t)cc));
                                if (NB == 2)
                                    st_async_f32(map_to_cta(dst + 128 * 4, (uint32_t)cc), p1, map_to_cta(bar_hid, (uint32_t)cc));
                            }
                        }
                    }
                    mbar_wait_cluster(bar_hid, (uint32_t)n_se & 1u);
                    {
                        const int j = tid;
#pragma unroll
                        for (int b = 0; b < NB; b++) {
                            const float *p = s_hidp + b * 128 + j;  // chunk k at p[k * 256]
                            s_hid[b * 128 + j] = se_hidden(se_b1v, se_tree4(p[0], p[256], p[512], p[768]),
                                                           se_tree4(p[1024], p[1280], p[1536], p[1792]));
                        }
                    }
                    lat_epi_sync();
                    // ---- FC2: one 32-hidden-unit chain per (board, channel, chunk), spread over the 128 threads ----
#pragma unroll
                    for (int i = 0; i < NB * NC * 4 / 128; i++) {
                        const int id = tid + 128 * i, o = id >> 2, k = id & 3;
                        const int b = o / NC, c = o % NC;
                        float acc = 0.f;
#pragma unroll
                        for (int qq = 0; qq < 4; qq++) {
                            const int q = 4 * k + qq;
                            float wf[8];
                            OT::unpack8(s_w2s[q * NC + c], wf);
                            acc = se_chain8(wf, *reinterpret_cast<const float4 *>(s_hid + b * 128 + q * 8),
                                            *reinterpret_cast<const float4 *>(s_hid + b * 128 + q * 8 + 4), acc);
                        }
                        s_fc2p[o * 4 + k] = acc;
                    }
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_sewe);  // the SE weight buffers may be refilled
                    lat_epi_sync();
                    if (tid < NB * NC) {
                        const float *c4 = s_fc2p + tid * 4;
                        s_gate[tid] = se_sigmoid(se_fc2_sum(se_b2v, c4[0], c4[1], c4[2], c4[3]));
                    }
                    lat_epi_sync();
                    n_se++;
                }
                if (prof) pe_se += clock64() - tq0;
                // ---- out = relu(gate * OT(y) + x), in place over the block input (y parked in the operand type, as the
                //      throughput kernel parks it in shared memory) ----
                if (active) {
                    const float *gate = s_gate + board * NC;
#pragma unroll
                    for (int i = 0; i < NC / 8; i++) {
                        const uint32_t xw[4] = {xres[i].x, xres[i].y, xres[i].z, xres[i].w};
                        uint32_t pw[4];
#pragma unroll
                        for (int k = 0; k < 4; k++) {
                            const int c = 8 * i + 2 * k;
                            const float yb0 = OT::round(a[c]);
                            const float yb1 = OT::round(a[c + 1]);
                            const float g0 = L.se == 1 ? gate[c] : 1.f, g1 = L.se == 1 ? gate[c + 1] : 1.f;
                            const float o0 = fmaxf(fmaf(g0, yb0, OT::lo(xw[k])), 0.f);
                            const float o1 = fmaxf(fmaf(g1, yb1, OT::hi(xw[k])), 0.f);
                            pw[k] = OT::pack2(o0, o1);
                        }
                        odst[i] = make_uint4(pw[0], pw[1], pw[2], pw[3]);
                    }
                }
            }
            // ---- hand the layer's output to the TMA loads of the whole cluster: every thread makes its staging-tile
            //      stores visible to the async proxy, block barrier, then ONE warp stores the CTA's slice and signals
            //      the `ready` barrier of every CTA ----
            const long long tf0 = prof ? clock64() : 0;
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            const long long tf1 = prof ? clock64() : 0;
            lat_epi_sync();
            const long long tf2 = prof ? clock64() : 0;
            if (quad == 0) {
                // one thread stores the CTA's slice and waits until the write is complete, then the warp signals
                if (elect_one()) {
                    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                                     NB == 2 ? &L.map_o : &L.map_o1),
                                 "r"(smem_base + (uint32_t)Cfg::OFF_OUT), "r"(c0), "r"(0), "r"(tile * NB), "r"(0)
                                 : "memory");
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
                }
                __syncwarp();
            }
            if (quad == 0 && lane < CL) mbar_arrive_cluster(map_to_cta(bar_ready, (uint32_t)lane));
            if (prof) {
                pe_pfence += tf1 - tf0;
                pe_sync += tf2 - tf1;
                pe_gfence += clock64() - tf2;
                pe_work += clock64() - tp1;
            }
        }
        if (prof) {
            args.prof[blockIdx.x * 16 + 6] = pe_tfull;
            args.prof[blockIdx.x * 16 + 7] = pe_stat;
            args.prof[blockIdx.x * 16 + 8] = pe_se;
            args.prof[blockIdx.x * 16 + 9] = pe_work;
            args.prof[blockIdx.x * 16 + 10] = pe_ld;
            args.prof[blockIdx.x * 16 + 11] = pe_pfence;
            args.prof[blockIdx.x * 16 + 12] = pe_sync;
            args.prof[blockIdx.x * 16 + 13] = pe_gfence;
        }
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();  // no CTA leaves while a peer may still signal it
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                     "r"((uint32_t)(NC < 32 ? 32 : NC))
                     : "memory");
    }
}

// ---- host side ------------------------------------------------------------------------------------------------
template <int CL> constexpr int lat_smem_bytes()
{
    return LatCfg<CL, 1>::SMEM_BYTES > LatCfg<CL, 2>::SMEM_BYTES ? LatCfg<CL, 1>::SMEM_BYTES : LatCfg<CL, 2>::SMEM_BYTES;
}

struct LatTower {
    LatLayer *d_layers[2] = {nullptr, nullptr};  // [0]: CL = 8, [1]: CL = 4
    int n_layers = 0;
    TcOp op = TC_OP_BF16;                        // TC_OP_BF16 (OpBf16) or TC_OP_FP16 (OpFp16)
    int max_tiles[2] = {0, 0};                   // co-resident clusters of 8 / 4 CTAs
    bool one_board = true;                       // one-board tiles (M64) while there are clusters for them
};

template <int CL, class OT> static int lat_max_clusters(int *out)
{
    SCB_CUDA(cudaFuncSetAttribute(lat_tower_kernel<CL, 2, OT>, cudaFuncAttributeMaxDynamicSharedMemorySize, lat_smem_bytes<CL>()));
    SCB_CUDA(cudaFuncSetAttribute(lat_tower_kernel<CL, 1, OT>, cudaFuncAttributeMaxDynamicSharedMemorySize, lat_smem_bytes<CL>()));
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(CL * 64);
    cfg.blockDim = dim3(LAT_THREADS);
    cfg.dynamicSmemBytes = lat_smem_bytes<CL>();
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CL;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int n = 0;
    SCB_CUDA(cudaOccupancyMaxActiveClusters(&n, lat_tower_kernel<CL, 2, OT>, &cfg));
    *out = n;
    return SC_OK;
}

int lat_tower_create(LatTower **out, const LatLayerDesc *descs, int n, int boards_alloc, TcOp op)
{
    if (op != TC_OP_BF16 && op != TC_OP_FP16) {
        set_error("lat_tower_create: no latency kernel for this operand type");
        return SC_E_INVAL;
    }
    const bool fp16 = op == TC_OP_FP16;
    LatTower *t = new LatTower();
    t->n_layers = n;
    t->op = op;
    const CUtensorMapDataType dt = fp16 ? OpFp16::TMAP : OpBf16::TMAP;
    for (int v = 0; v < 2; v++) {
        const int CL = v == 0 ? 8 : 4, NC = 256 / CL;
        std::vector<LatLayer> h((size_t)n);
        for (int i = 0; i < n; i++) {
            const LatLayerDesc &d = descs[i];
            LatLayer &L = h[i];
            memset(&L, 0, sizeof(L));
            int rc = tc_make_act_map_hbw(dt, d.in, boards_alloc, d.cin_pad, &L.map_a);
            if (rc == SC_OK) {
                // the same tensor {C, file, board, rank} with a box of ONE board: 80 rows ordered (rank, file)
                cuuint64_t dims[4] = {(cuuint64_t)d.cin_pad, 8, (cuuint64_t)boards_alloc, 8};
                cuuint64_t strides[3] = {(cuuint64_t)d.cin_pad * 2, (cuuint64_t)d.cin_pad * 128, (cuuint64_t)d.cin_pad * 16};
                cuuint32_t box[4] = {TC_BK, 8, 1, 10};
                rc = tc_encode_map(&L.map_a1, dt, d.in, 4, dims, strides, box, "activations (rank, file), one board");
            }
            if (rc == SC_OK) {
                // output {C, file, board, rank}: box of this CTA's NC channels of the tile's boards, unswizzled
                cuuint64_t dims[4] = {256, 8, (cuuint64_t)boards_alloc, 8};
                cuuint64_t strides[3] = {256 * 2, 256 * 128, 256 * 16};
                cuuint32_t box2[4] = {(cuuint32_t)NC, 8, 2, 8}, box1[4] = {(cuuint32_t)NC, 8, 1, 8};
                rc = tc_encode_map(&L.map_o, dt, d.out, 4, dims, strides, box2, "output slice, two boards", false);
                if (rc == SC_OK) rc = tc_encode_map(&L.map_o1, dt, d.out, 4, dims, strides, box1, "output slice, one board", false);
            }
            if (rc == SC_OK) {
                // weights [tap = dy * 3 + dx][256][cin_pad] as {cin, cout, dx, dy}
                const int nd = d.taps == 9 ? 3 : 1;
                cuuint64_t dims[4] = {(cuuint64_t)d.cin_pad, 256, (cuuint64_t)nd, (cuuint64_t)nd};
                cuuint64_t strides[3] = {(cuuint64_t)d.cin_pad * 2, (cuuint64_t)d.cin_pad * 2 * 256,
                                         (cuuint64_t)d.cin_pad * 2 * 256 * 3};
                cuuint32_t box[4] = {TC_BK, (cuuint32_t)NC, 1, (cuuint32_t)nd};
                rc = tc_encode_map(&L.map_w, dt, d.w, 4, dims, strides, box, "weights (cluster slice)");
            }
            if (rc != SC_OK) {
                lat_tower_destroy(t);
                return rc;
            }
            L.resid = d.resid;
            L.bias = d.bias;
            L.gamma = d.gamma;
            L.beta = d.beta;
            L.se_w1s = static_cast<const uint4 *>(v == 0 ? d.se_w1s8 : d.se_w1s4);
            L.se_w2s = static_cast<const uint4 *>(v == 0 ? d.se_w2s8 : d.se_w2s4);
            L.se_b1 = d.se_b1;
            L.se_b2 = d.se_b2;
            L.taps = d.taps;
            L.kchunks = d.cin_pad / TC_BK;
            L.relu = d.relu;
            L.se = d.se;
            L.ln = d.ln;
            if (d.se && !d.resid) {
                set_error("lat_tower_create: residual layer without block input");
                lat_tower_destroy(t);
                return SC_E_INVAL;
            }
        }
        if (cudaMalloc(&t->d_layers[v], sizeof(LatLayer) * (size_t)n) != cudaSuccess ||
            cudaMemcpy(t->d_layers[v], h.data(), sizeof(LatLayer) * (size_t)n, cudaMemcpyHostToDevice) != cudaSuccess) {
            lat_tower_destroy(t);
            set_error("lat_tower_create: device allocation failed");
            return SC_E_CUDA;
        }
    }
    int rc = fp16 ? lat_max_clusters<8, OpFp16>(&t->max_tiles[0]) : lat_max_clusters<8, OpBf16>(&t->max_tiles[0]);
    if (rc == SC_OK) rc = fp16 ? lat_max_clusters<4, OpFp16>(&t->max_tiles[1]) : lat_max_clusters<4, OpBf16>(&t->max_tiles[1]);
    if (rc != SC_OK) {
        lat_tower_destroy(t);
        return rc;
    }
    if (getenv("SCB200_LAT_CLUSTER")) {  // A/B: force one cluster size
        const int want = atoi(getenv("SCB200_LAT_CLUSTER"));
        if (want == 4) t->max_tiles[0] = 0;
        if (want == 8) t->max_tiles[1] = 0;
    }
    t->one_board = !(getenv("SCB200_LAT_ONE_BOARD") && getenv("SCB200_LAT_ONE_BOARD")[0] == '0');  // A/B
    *out = t;
    return SC_OK;
}

void lat_tower_destroy(LatTower *t)
{
    if (!t) return;
    for (int v = 0; v < 2; v++)
        if (t->d_layers[v]) cudaFree(t->d_layers[v]);
    delete t;
}

int lat_tower_max_boards(const LatTower *t) { return t ? 2 * (t->max_tiles[0] > t->max_tiles[1] ? t->max_tiles[0] : t->max_tiles[1]) : 0; }

template <int CL, int NB, class OT> static int lat_launch(const LatTower *t, int v, int n_tiles, cudaStream_t st, int max_layers)
{
    LatArgs a;
    a.layers = t->d_layers[v];
    a.n_layers = max_layers > 0 && max_layers < t->n_layers ? max_layers : t->n_layers;
    a.n_tiles = n_tiles;
    a.prof = nullptr;
    static const bool want_prof = getenv("SCB200_PHASE_PROFILE") != nullptr;
    if (want_prof) {
        SCB_CUDA(cudaMalloc(&a.prof, (size_t)n_tiles * CL * 16 * sizeof(long long)));
        SCB_CUDA(cudaMemsetAsync(a.prof, 0, (size_t)n_tiles * CL * 16 * sizeof(long long), st));
    }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(n_tiles * CL);
    cfg.blockDim = dim3(LAT_THREADS);
    cfg.dynamicSmemBytes = lat_smem_bytes<CL>();
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CL;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    SCB_CUDA(cudaLaunchKernelEx(&cfg, lat_tower_kernel<CL, NB, OT>, a));
    SCB_CUDA(cudaGetLastError());
    if (want_prof) {
        // debugging aid (synchronous): SM cycles per phase, summed over the layers, averaged over the CTAs
        std::vector<long long> h((size_t)n_tiles * CL * 16);
        SCB_CUDA(cudaStreamSynchronize(st));
        SCB_CUDA(cudaMemcpy(h.data(), a.prof, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
        cudaFree(a.prof);
        double acc[16] = {0};
        for (int b = 0; b < n_tiles * CL; b++)
            for (int k = 0; k < 16; k++) acc[k] += (double)h[(size_t)b * 16 + k] / (n_tiles * CL);
        fprintf(stderr,
                "[lat CL=%d NB=%d tiles=%d layers=%d] A-producer: wait_ready %.0f wait_empty %.0f | mma: total %.0f wait_A(first box) %.0f "
                "wait(rest) %.0f (%.0f) | epilogue: wait_tmem_full %.0f work %.0f (tmem load %.0f, stat exchange %.0f, SE %.0f, "
                "proxy fence %.0f, block barrier %.0f, TMA store + signal %.0f)\n",
                CL, NB, n_tiles, a.n_layers, acc[0], acc[1], acc[5], acc[2], acc[3], acc[4], acc[6], acc[9], acc[10], acc[7], acc[8],
                acc[11], acc[12], acc[13]);
    }
    return SC_OK;
}

template <class OT> static int lat_dispatch(const LatTower *t, int n_boards, cudaStream_t st, int max_layers)
{
    const int n_tiles = (n_boards + 1) / 2;
    if (t->one_board && n_boards <= t->max_tiles[0]) return lat_launch<8, 1, OT>(t, 0, n_boards, st, max_layers);
    if (t->one_board && n_boards <= t->max_tiles[1]) return lat_launch<4, 1, OT>(t, 1, n_boards, st, max_layers);
    if (n_tiles <= t->max_tiles[0]) return lat_launch<8, 2, OT>(t, 0, n_tiles, st, max_layers);
    if (n_tiles <= t->max_tiles[1]) return lat_launch<4, 2, OT>(t, 1, n_tiles, st, max_layers);
    return SC_E_STATE;
}

// SC_E_STATE (no message): the batch does not fit one wave of clusters; the caller runs the throughput kernel
int lat_tower_launch(LatTower *t, int n_boards, cudaStream_t st, int max_layers)
{
    if (n_boards <= 0) return SC_OK;
    // one-board tiles (half the operand traffic per CTA) while every board can have a cluster -- 8 CTAs per board, then 4
    // (measured, n = 16: 0.418 ms against 0.433 ms for two boards per 8-CTA cluster) -- then two-board tiles
    return t->op == TC_OP_FP16 ? lat_dispatch<OpFp16>(t, n_boards, st, max_layers)
                               : lat_dispatch<OpBf16>(t, n_boards, st, max_layers);
}

}  // namespace scb
