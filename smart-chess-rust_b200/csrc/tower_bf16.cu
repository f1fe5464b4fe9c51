// bf16 throughput mode of the policy/value network: tcgen05 / TMEM / TMA implicit-GEMM
// convolutions with bias + LayerNorm(C) (+ReLU | + squeeze-excitation + residual + ReLU)
// fused into the epilogue, for sm_100a.
//
// Network arithmetic restated from py/module.py:120-126 (stem), :38-46 (ResBlockSE),
// :70-76 / :89-93 (head 1x1 convs); LayerNorm2d = LN over channels, eps 1e-6 (timm);
// SqueezeExcitation(256, 128) = sigmoid(fc2(relu(fc1(avgpool)))) * x (torchvision).
//
// GEMM view of one 3x3 layer: M = 64 * boards, N = 256 output channels, K = 9 taps x Cin.
//   A (activations, bf16 NHWC [board][rank][file][C]) is never materialised as im2col.  The 256-wide
//   convolutions (pair kernels): ONE box {64 ch, 8 files, 2 boards, 10 ranks} at (64*kc, dx, board0, -1)
//   serves the three dy taps of channel chunk kc and column shift dx; it lands as 160 rows ordered
//   (rank, board, file) and tap dy is the 128-row tile 2 KB * (dy + 1) into it.  The policy head (a
//   single-CTA 1x1 convolution) loads the 4-D box {64 ch, 8 files, 8 ranks, 2 boards} at (64*kc, 0, 0, board0).
//   Ranks/files outside [0,8) are zero-filled by the TMA unit, which IS the conv padding; 128B swizzle
//   makes every tile the canonical K-major UMMA operand.
//   B (weights, bf16 [tap][cout][cin]) is a plain 2-D box.
//   D accumulates in TMEM (128 lanes x 256 fp32 columns per tile, two tiles = all 512
//   columns, so the epilogue of tile i overlaps the MMAs of tile i+1).
// One kernel template, tc_gemm_kernel<BN, EPI, A4D, CTA2, TOWER, OT>:
//   * OT: the operand type, OpBf16, OpFp16 or OpE4m3 (tc_ptx.cuh).  Activations, weights and the stored layer outputs
//     are of that type, the parked SE tile of OT::Park; the accumulator, LayerNorm, SE arithmetic and the head tails are
//     fp32.  OpE4m3's K chunk is 128 channels (OT::BK), the same 128 bytes as 64 16-bit channels, and its epilogues
//     apply the per-channel weight scale first (acc * scale + bias);
//   * CTA2: every 256-wide convolution; clusters of two CTAs issue tcgen05.mma.cta_group::2 (256-row
//     tiles, each CTA stages its own rows of A and half of the weight rows);
//   * TOWER: the stem, all residual blocks and the two 256-wide head 1x1 convolutions run
//     in ONE persistent launch; a tile's layers are chained by a per-tile mbarrier inside
//     the CTA (boards never interact inside the tower), tiles are carried through all
//     layers in groups of 3-4 so that layer outputs are re-read from L2;
//   * the narrow head GEMMs (256->73 with LayerNorm(73), optionally followed in the same epilogue
//     by log-softmax + legal-move gather + renormalisation; value FC 16384->128 as a split-K
//     GEMM whose rows are boards) are the single-CTA instantiations of the same kernel.
// Producer and MMA warps run warp-uniform loops and elect one lane around the TMA / MMA / commit
// instructions only, which keeps descriptors and barrier addresses in uniform registers.
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer,
// warps 2..9 = epilogue (two warps per TMEM lane quadrant, each owning 128 of the 256
// columns of its 32 rows; one thread = one (board, square) row, so LayerNorm over channels
// is a per-thread reduction plus one exchange with the sibling warp).
#include <cuda.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <type_traits>
#include <vector>

#include "common.cuh"
#include "move_index.cuh"

#include "tc_ptx.cuh"
#include "tc_host.cuh"

namespace scb {

constexpr int TC_BN = 256;
constexpr int TC_STAGES = 4;
constexpr int TC_A_BYTES = TC_BM * TC_BK * 2;  // 16 KB
constexpr int TC_THREADS = 320;      // warp 0 TMA, warp 1 MMA, warps 2..9 epilogue (two per TMEM lane quadrant)

// ---- the kernel ---------------------------------------------------------------------------
// Epilogue variants of the one warp-specialised GEMM kernel:
//   EPI_LN     bias + LayerNorm(256) (+ReLU)                     -> bf16 [rows][256]
//   EPI_LN_SE  bias + LayerNorm(256) + squeeze-excitation + residual + ReLU, all inside the
//              epilogue (a tile is two whole boards, so the SE average pool is a reduction
//              over the tile's own rows)                          -> bf16 [rows][256]
//   EPI_LN73   bias + LayerNorm(73) of the 80-wide policy map     -> fp32 [rows][80]
//   EPI_RAW    split-K partial sums of the value FC               -> fp32 [split][M][128]
//   EPI_LN73_GATHER  EPI_LN73, but the 64 x 73 logits of a leaf stay in shared memory: log-softmax over the
//              4672 entries, gather at the legal moves' indices, renormalise            -> priors
//   EPI_F32    bias only, fp32 accumulator out                    -> fp32 [rows][256]   (FP32 parity mode: the GEMM
//              runs the bf16x3 operand split, LayerNorm / SE follow in tower_f32.cu's fp32 kernels)
enum { EPI_LN = 0, EPI_LN_SE = 1, EPI_LN73 = 2, EPI_RAW = 3, EPI_LN73_GATHER = 4, EPI_F32 = 5 };

// One convolution layer of the whole-tower kernel (device array, written once at engine creation)
struct alignas(64) TowerLayer {
    CUtensorMap map_a;                   // activations of the layer's input buffer (4-D, box of two boards)
    CUtensorMap map_w;                   // this layer's weights, box {64, 128} (one CTA's half)
    void *out;
    const __nv_bfloat16 *resid;
    const float *bias, *gamma, *beta;
    const uint4 *se_w1p, *se_w2p;
    const float *se_b1, *se_b2;
    int taps, kchunks, relu, se;
    int ln;                              // 0: no LayerNorm (BatchNorm folded at export): y = acc + bias
    const float *scale;                  // scaled operand types (OpE4m3): per-channel weight scales, y = acc * scale + bias
};

struct TcArgs {
    void *out;
    const __nv_bfloat16 *resid;          // EPI_LN_SE: block input x (may alias out)
    const float *bias, *gamma, *beta;
    const uint4 *se_w1p, *se_w2p;        // EPI_LN_SE: fc1 as [32][128][8] bf16, fc2 as [16][256][8] bf16
    const float *se_b1, *se_b2;
    int n_tiles;                         // M tiles of 128 rows
    int taps, kchunks;                   // k-blocks per work item = taps * kchunks
    int relu;
    int ln;                              // 0: the layer has no LayerNorm (y = acc + bias)
    int n_splits;                        // EPI_RAW: work items = n_tiles * n_splits
    int m_rows;                          // EPI_RAW: valid rows
    // FP32 parity mode (bf16x3 split): an fp32 product a * b is the sum of bf16 products a_i * b_j of the operands'
    // three bf16 planes (a = a_0 + a_1 + a_2, |a_k| ~ 2^-8k |a|); the planes are concatenated along the channel
    // dimension of both tensors and the k loop walks `split_pairs` (A plane, B plane) pairs of `split_kreal` channel
    // chunks each, smallest terms first, all into the same fp32 accumulator.  0 = plain bf16 GEMM.
    int split_pairs, split_kreal;
    uint8_t split_ap[8], split_bp[8];
    long long *prof;                     // optional [grid][16] phase cycle counters (SCB200_PHASE_PROFILE=1)
    const TowerLayer *layers;            // TOWER: all conv layers of the residual tower, run back to back
    int n_layers;
    int group;                           // TOWER: tiles per CTA carried through all layers together (0 = all)
    TcGather gather;                     // EPI_LN73_GATHER: legal moves in, priors out
    TcValueFinish vfin;                  // EPI_RAW: value head tail fused into the split-K GEMM (counters != nullptr)
    const float *scale;                  // scaled operand types: per-output-channel weight scales (EPI_RAW: of the
                                         // hidden units, applied after the split sum)
};

__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }
// EPI_LN73_GATHER: one barrier per set of four epilogue warps (set 0 = warps 2..5, set 1 = warps 6..9)
__device__ __forceinline__ void gather_bar_sync(int set) { asm volatile("bar.sync %0, 128;" ::"r"(2 + set) : "memory"); }

// Per-warp staging tile of 32 rows x 64 bytes used to turn the epilogue's thread-per-row data
// into coalesced global accesses (a row-per-lane access has a 512-byte lane stride and costs 32
// half-used sectors per instruction; through the tile every instruction covers 8 rows x 64 B =
// 16 full sectors).  16-byte chunk q of row r lives at chunk q ^ ((r >> 1) & 3): conflict-free
// for both the row-per-lane and the 4-lanes-per-row access.
__device__ __forceinline__ uint32_t stg_off(int row, int q) { return (uint32_t)(row * 64 + ((q ^ ((row >> 1) & 3)) << 4)); }

// lane's own 64 bytes (row = lane) -> staging -> global rows gbase + r * row_stride (+ 16-byte chunk)
__device__ __forceinline__ void staged_store_64B(uint8_t *stg, int lane, const uint4 (&v)[4], uint8_t *gbase,
                                                 size_t row_stride, int rows_valid)
{
#pragma unroll
    for (int q = 0; q < 4; q++) *reinterpret_cast<uint4 *>(stg + stg_off(lane, q)) = v[q];
    __syncwarp();
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int rr = (lane >> 2) + 8 * k;
        const uint4 t = *reinterpret_cast<const uint4 *>(stg + stg_off(rr, lane & 3));
        if (rr < rows_valid) *reinterpret_cast<uint4 *>(gbase + (size_t)rr * row_stride + (lane & 3) * 16) = t;
    }
    __syncwarp();
}

// Same, for accumulator rows ordered (rank, board, file) (pair kernels, shared activation box): the warp of
// TMEM quadrant `quad` holds ranks 2 quad and 2 quad + 1 of both boards; its 8-row group k is rank 2 quad + k / 2
// of board k % 2, i.e. tile rows 64 (k % 2) + 8 (2 quad + k / 2) .. + 7 in memory.
__device__ __forceinline__ void staged_store_64B_hbw(uint8_t *stg, int lane, const uint4 (&v)[4], uint8_t *tile_base,
                                                     size_t row_stride, int quad)
{
#pragma unroll
    for (int q = 0; q < 4; q++) *reinterpret_cast<uint4 *>(stg + stg_off(lane, q)) = v[q];
    __syncwarp();
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int rr = (lane >> 2) + 8 * k;
        const uint4 t = *reinterpret_cast<const uint4 *>(stg + stg_off(rr, lane & 3));
        const int grow = (k & 1) * 64 + (quad * 2 + (k >> 1)) * 8 + (lane >> 2);
        *reinterpret_cast<uint4 *>(tile_base + (size_t)grow * row_stride + (lane & 3) * 16) = t;
    }
    __syncwarp();
}

template <int BN, bool CTA2 = false, bool YSMEM = false> struct TcCfg {
    // single CTA (the narrow heads): one ring of stages, each holding an A tile and a B tile
    static constexpr int STAGES = TC_STAGES;
    // cta_group::2: the pair computes a 256-row tile; each CTA stages its own 128 rows of A and HALF of the weight rows.
    // The three dy taps of a (channel chunk, dx) read ONE activation box of 10 board rows (rank -1..8, zero-filled
    // outside the board) instead of three boxes of 8: separate rings for the 20 KB activation boxes (NA) and the 16 KB
    // weight tiles (NB), 29 % fewer bytes from L2 per tile.  The SE variant gives up ring slots for a 64 KB bf16 copy of
    // the tile's LayerNorm output (YSMEM), see the epilogue.
    static constexpr int NA = YSMEM ? 3 : 4, NB = YSMEM ? 4 : 7;
    static constexpr int A_BOX_BYTES = 160 * TC_BK * 2;  // rows ordered (rank, board, file): 10 x 2 x 8
    // BN == LD_POLICY: room for the fp32 logits of the tile's two leaves ([128][81], odd row stride = no bank
    // conflicts), the unnormalised priors of both leaves and the cross-warp reductions (EPI_LN73_GATHER)
    static constexpr int G_BYTES = BN == LD_POLICY ? 2 * (TC_BM * 81 + 2 * SC_MAX_MOVES + 16) * 4 : 0;  // two warp sets
    static constexpr int Y_BYTES = YSMEM ? TC_BM * 256 * 2 : G_BYTES;
    static constexpr int B_BYTES = (CTA2 ? BN / 2 : BN) * TC_BK * 2;
    static constexpr int STAGE_BYTES = TC_A_BYTES + B_BYTES;
    static constexpr int SMEM_EPI = 3 * 256 * 4 /*bias,gamma,beta*/ + (4 * 256 /*unused*/ + 2 * 256 + 2 * 128 + 2 * 256) * 4 /*SE*/ +
                                    (2 * 256 + 4 * 128) * 4 /*LN partials, FC1 partials*/ + 8 * 2048 /*store staging*/;
    static constexpr int RING_BYTES = CTA2 ? NA * A_BOX_BYTES + NB * B_BYTES : STAGES * STAGE_BYTES;
    static constexpr int N_RING_BARS = CTA2 ? 2 * (NA + NB) : 2 * STAGES;
    static constexpr int SMEM_BYTES = RING_BYTES + SMEM_EPI + Y_BYTES + 768;
};

constexpr int TC_MAX_SLOTS = 32;  // TOWER: tiles per CTA whose layer-to-layer hand-over is tracked

template <int BN, int EPI, bool A4D, bool CTA2 = false, bool TOWER = false, class OT = OpBf16>
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w,
               const TcArgs args)
{
    // TOWER: one launch runs every convolution of the residual tower.  Boards never interact inside the
    // tower, so layer l+1 of a tile depends only on layer l of the SAME tile, which the same CTA
    // produced: the hand-over is a per-tile mbarrier inside the CTA, there is no grid-wide barrier, no
    // per-layer launch gap and no per-layer tail.
    static_assert(!TOWER || (CTA2 && EPI == EPI_LN_SE), "tower kernel = pair mode with both epilogues compiled in");
    static_assert(EPI != EPI_F32 || std::is_same<OT, OpBf16>::value, "the bf16x3 split of the FP32 parity mode is bf16");
    constexpr bool YSMEM = EPI == EPI_LN_SE;
    using Cfg = TcCfg<BN, CTA2, YSMEM>;
    constexpr int STAGE_BYTES = Cfg::STAGE_BYTES;
    constexpr int NSTAGES = Cfg::STAGES;
    static_assert(!CTA2 || (A4D && BN == 256 && (EPI == EPI_LN || EPI == EPI_LN_SE || EPI == EPI_F32)),
                  "pair mode: tower convs only");
    static_assert(CTA2 || ((BN == LD_POLICY && (EPI == EPI_LN73 || EPI == EPI_LN73_GATHER)) || (BN == N_VALUE_HIDDEN && EPI == EPI_RAW)),
                  "single CTA: narrow head GEMMs only");
    const uint32_t cta_rank = CTA2 ? __shfl_sync(0xffffffffu, cluster_ctarank(), 0) : 0u;
    const int work0 = CTA2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int work_stride = CTA2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    // Dynamic shared memory is the only shared allocation of this kernel, so it starts at offset 0 of
    // the CTA window and is 1024-byte aligned (required by the 128B swizzle); checked below.  Deriving
    // the pointers directly from the __shared__ symbol keeps every access an LDS/STS (a pointer
    // laundered through an integer cast degrades to generic LD/ST).
    extern __shared__ __align__(1024) uint8_t smem[];
    constexpr int NA = Cfg::NA, NB = Cfg::NB, A_BOX = Cfg::A_BOX_BYTES, B_TILE = Cfg::B_BYTES;
    constexpr int NRB = Cfg::N_RING_BARS;
    float *s_bias = reinterpret_cast<float *>(smem + Cfg::RING_BYTES);
    float *s_gamma = s_bias + 256;
    float *s_beta = s_gamma + 256;
    float *s_scale = s_beta + 256;        // OT::SCALED: the weight scales [256] (the 4 KB up to s_mean are otherwise unused)
    float *s_mean = s_beta + 256 + 1024;  // [2 boards][256]
    float *s_hid = s_mean + 512;    // [2][128]
    float *s_gate = s_hid + 256;    // [2][256]
    float *s_stat = s_gate + 512;   // [2 column halves][128 rows][sum, sumsq]
    float *s_hidp = s_stat + 512;   // [2 channel halves][2 boards][128]
    uint8_t *s_stage = reinterpret_cast<uint8_t *>(s_hidp + 512);  // [8 epilogue warps][32 rows][64 B]
    uint8_t *s_y = s_stage + 8 * 2048;  // YSMEM: [128 rows][32 chunks of 16 B], chunk index XOR (row & 7)
    uint64_t *bars = reinterpret_cast<uint64_t *>(s_y + Cfg::Y_BYTES);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + NRB + 4 + TC_MAX_SLOTS);

    // warp index and CTA rank as warp-uniform values: the producer and MMA warps run their loops with all 32 lanes
    // and elect one lane only around the TMA / tcgen05 instructions, so descriptors, barrier addresses and
    // coordinates live in uniform registers instead of being broadcast lane -> uniform before every instruction
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const uint32_t smem_base = smem_u32(smem);
    if (smem_base & 1023u) __trap();
    const uint32_t bar_base = smem_u32(bars);
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (NSTAGES + s); };
    auto tfull_bar = [&](int s) { return bar_base + 8u * (NRB + s); };
    auto tempty_bar = [&](int s) { return bar_base + 8u * (NRB + 2 + s); };
    auto ready_bar = [&](int s) { return bar_base + 8u * (NRB + 4 + s); };  // TOWER: tile s written by layer l
    // pair rings: activation boxes first, then weight tiles
    auto afull_bar = [&](int s) { return bar_base + 8u * s; };
    auto aempty_bar = [&](int s) { return bar_base + 8u * (NA + s); };
    auto bfull_bar = [&](int s) { return bar_base + 8u * (2 * NA + s); };
    auto bempty_bar = [&](int s) { return bar_base + 8u * (2 * NA + NB + s); };
    auto abox_addr = [&](int s) { return smem_base + (uint32_t)(s * A_BOX); };
    auto btile_addr = [&](int s) { return smem_base + (uint32_t)(NA * A_BOX + s * B_TILE); };

    struct LayerView {
        const CUtensorMap *ma, *mw;
        void *out;
        const __nv_bfloat16 *resid;
        const float *bias, *gamma, *beta;
        const uint4 *w1p, *w2p;
        const float *b1, *b2;
        int taps, kchunks, relu;
        bool se, ln;
        bool se_fc;  // se: squeeze-excitation gate (false with se: residual + ReLU only, `use_se=False`)
        const float *scale;
    };
    auto layer_view = [&](int l) -> LayerView {
        if constexpr (TOWER) {
            const TowerLayer &T = args.layers[l];
            return LayerView{&T.map_a, &T.map_w, T.out, T.resid, T.bias, T.gamma, T.beta, T.se_w1p, T.se_w2p, T.se_b1, T.se_b2,
                             T.taps, T.kchunks, T.relu, T.se != 0, T.ln != 0, T.se == 1, OT::SCALED ? T.scale : nullptr};
        } else {
            return LayerView{&map_a, &map_w, args.out, args.resid, args.bias, args.gamma, args.beta, args.se_w1p, args.se_w2p,
                             args.se_b1, args.se_b2, args.taps, args.kchunks, args.relu, EPI == EPI_LN_SE, args.ln != 0,
                             EPI == EPI_LN_SE && args.se_w1p != nullptr, OT::SCALED ? args.scale : nullptr};
        }
    };
    // a = acc + bias of channel c (scaled types: acc * scale + bias; the scale is a power of two, so the product is exact
    // and the fma rounds once, like the add)
    auto acc_bias = [&](uint32_t acc, int c) -> float {
        if constexpr (OT::SCALED) return __fmaf_rn(__uint_as_float(acc), s_scale[c], s_bias[c]);
        else return __fadd_rn(__uint_as_float(acc), s_bias[c]);
    };
    // the same for the narrow head epilogues, whose unscaled form is a contractible add
    auto head_a = [&](uint32_t acc, int c) -> float {
        if constexpr (OT::SCALED) return __fmaf_rn(__uint_as_float(acc), s_scale[c], s_bias[c]);
        else return __uint_as_float(acc) + s_bias[c];
    };
    const int n_layers = TOWER ? args.n_layers : 1;

    if (EPI != EPI_RAW && !TOWER) {
        constexpr int NV = (EPI == EPI_LN73 || EPI == EPI_LN73_GATHER) ? C_POLICY : BN;
        for (int i = threadIdx.x; i < 256; i += TC_THREADS) {
            s_bias[i] = i < NV ? args.bias[i] : 0.f;
            s_gamma[i] = i < NV ? (args.ln ? args.gamma[i] : 1.f) : 0.f;
            s_beta[i] = i < NV && args.ln ? args.beta[i] : 0.f;
            if constexpr (OT::SCALED) s_scale[i] = i < NV ? args.scale[i] : 0.f;
        }
    }
    if (threadIdx.x == 0) {
        for (int s = 0; s < NRB; s++) mbar_init(bar_base + 8u * s, 1);  // ring barriers: one producer / one commit each
        if (TOWER)
            for (int s = 0; s < TC_MAX_SLOTS; s++) mbar_init(ready_bar(s), 256);
        for (int s = 0; s < 2; s++) {
            mbar_init(tfull_bar(s), 1);
            mbar_init(tempty_bar(s), ((EPI == EPI_LN || EPI == EPI_LN_SE || EPI == EPI_F32) ? 256 : 128) * (CTA2 ? 2 : 1));
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        if (CTA2) {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                         "r"(512u)
                         : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                         "r"(512u)
                         : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
    }
    tc_fence_before();
    __syncthreads();
    if (CTA2) cluster_sync_all();  // the peer's barriers are initialised before any remote arrive / complete_tx
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int n_work = EPI == EPI_RAW ? args.n_tiles * args.n_splits : (CTA2 ? (args.n_tiles + 1) / 2 : args.n_tiles);
    // This CTA's work items are visited group by group; a group of tiles goes through ALL layers before the
    // next group starts (TOWER), so a tile's output is re-read while it is still in L2.  Groups have >= 2 tiles
    // whenever possible: with the double-buffered accumulator the epilogue of one tile overlaps the MMAs of
    // the next tile of the group.  Outside the tower kernel there is one layer and one group.
    const int n_slots = work0 < n_work ? (n_work - work0 + work_stride - 1) / work_stride : 0;
    const int gsz_req = (TOWER && args.group > 0) ? args.group : (n_slots > 0 ? n_slots : 1);
    // ceil(n_slots / gsz_req): no group is larger than requested.  A group's activations (x and t of its tiles, 64 KB per
    // board) must stay in L2 next to the weights (52 MB) until the next layer has read them; at 2048 leaves a pair has 7
    // tiles: groups of (3, 4) = 76 MB of activations over the chip wrote 1.54 GB per launch back to DRAM, (2, 2, 3) writes
    // 0.47 GB and runs the power-capped SMs 4 % faster (profiles/r02_tile_groups.md)
    int n_groups = (n_slots + gsz_req - 1) / gsz_req;
    if (TOWER && args.group < 0) n_groups = -args.group;      // group < 0: that many groups per CTA pair (A/B runs)
    if (n_groups > n_slots) n_groups = n_slots;
    if (n_groups < 1) n_groups = 1;
    auto group_begin = [&](int gi) { return (int)(((long long)gi * n_slots) / n_groups); };

    if (warp == 0) {
        {
            if (lane == 0) {
                asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
                asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w) : "memory");
            }
            int stage = 0, astage = 0, bstage = 0;
            uint32_t phase = 0, aphase = 0, bphase = 0;
            long long pc_wait_empty = 0;
            for (int gi = 0; gi < n_groups; gi++)
            for (int layer = 0; layer < n_layers; layer++) {
            const LayerView P = layer_view(layer);
            for (int slot = group_begin(gi); slot < group_begin(gi + 1); slot++) {
                const int work = work0 + slot * work_stride;
                if (TOWER && layer > 0) mbar_wait(ready_bar(slot), (uint32_t)(layer - 1) & 1u);  // this tile's input is written
                const int tile = EPI == EPI_RAW ? work / args.n_splits : (CTA2 ? work * 2 + (int)cta_rank : work);
                const int split = EPI == EPI_RAW ? work % args.n_splits : 0;
                if constexpr (CTA2) {
                    const int nd = P.taps == 9 ? 3 : 1;
                    for (int kc = 0; kc < P.kchunks; kc++) {
                        // channel chunk of the A / B tensor this k step reads (the same one unless the operands are split)
                        int ca = kc, cb = kc;
                        if (!TOWER && args.split_pairs > 0) {
                            const int pr = kc / args.split_kreal, kk = kc % args.split_kreal;
                            ca = args.split_ap[pr] * args.split_kreal + kk;
                            cb = args.split_bp[pr] * args.split_kreal + kk;
                        }
                        for (int dxi = 0; dxi < nd; dxi++) {
                            const long long t0 = args.prof ? clock64() : 0;
                            mbar_wait(aempty_bar(astage), aphase ^ 1u);
                            if (args.prof) pc_wait_empty += clock64() - t0;
                            if (elect_one()) {
                                // both CTAs load into their own shared memory and complete on the LEADER's barrier,
                                // which the leader alone arms with the bytes of both
                                if (cta_rank == 0) mbar_expect_tx(afull_bar(astage), 2 * A_BOX);
                                tma2_load_4d(abox_addr(astage), P.ma, afull_bar(astage), ca * OT::BK, nd == 3 ? dxi - 1 : 0, tile * 2, -1);
                            }
                            __syncwarp();
                            for (int dyi = 0; dyi < nd; dyi++) {
                                const int tap = nd == 3 ? dyi * 3 + dxi : 0;
                                const long long t1 = args.prof ? clock64() : 0;
                                mbar_wait(bempty_bar(bstage), bphase ^ 1u);
                                if (args.prof) pc_wait_empty += clock64() - t1;
                                if (elect_one()) {
                                    if (cta_rank == 0) mbar_expect_tx(bfull_bar(bstage), 2 * B_TILE);
                                    tma2_load_2d(btile_addr(bstage), P.mw, bfull_bar(bstage), cb * OT::BK,
                                                 tap * BN + (int)cta_rank * (BN / 2));
                                }
                                __syncwarp();
                                if (++bstage == NB) {
                                    bstage = 0;
                                    bphase ^= 1u;
                                }
                            }
                            if (++astage == NA) {
                                astage = 0;
                                aphase ^= 1u;
                            }
                        }
                    }
                    continue;
                }
                for (int tap = 0; tap < P.taps; tap++) {
                    const int dy = P.taps == 9 ? tap / 3 - 1 : 0;
                    const int dx = P.taps == 9 ? tap % 3 - 1 : 0;
                    for (int kc = 0; kc < P.kchunks; kc++) {
                        const long long t0 = args.prof ? clock64() : 0;
                        mbar_wait(empty_bar(stage), phase ^ 1u);
                        if (args.prof) pc_wait_empty += clock64() - t0;
                        const uint32_t a_dst = smem_base + stage * STAGE_BYTES;
                        const uint32_t b_dst = a_dst + TC_A_BYTES;
                        if (!elect_one()) {
                        } else if (A4D) {
                            mbar_expect_tx(full_bar(stage), STAGE_BYTES);
                            tma_load_4d(a_dst, &map_a, full_bar(stage), kc * OT::BK, dx, dy, tile * 2);
                            tma_load_2d(b_dst, &map_w, full_bar(stage), kc * OT::BK, tap * BN);
                        } else {
                            mbar_expect_tx(full_bar(stage), STAGE_BYTES);
                            const int k0 = (split * P.kchunks + kc) * OT::BK;
                            tma_load_2d(a_dst, &map_a, full_bar(stage), k0, tile * TC_BM);
                            tma_load_2d(b_dst, &map_w, full_bar(stage), k0, 0);
                        }
                        if (++stage == NSTAGES) {
                            stage = 0;
                            phase ^= 1u;
                        }
                    }
                }
            }
            }
            if (args.prof && lane == 0) args.prof[blockIdx.x * 16 + 0] = pc_wait_empty;
        }
    } else if (warp == 1) {
        if (cta_rank == 0) {
            constexpr uint32_t idesc = umma_idesc<OT>(CTA2 ? 2 * TC_BM : TC_BM, BN);
            int stage = 0, ra = 0, rb = 0;
            uint32_t phase = 0, rap = 0, rbp = 0;
            int it = 0;
            long long pc_wait_tempty = 0, pc_wait_full = 0, pc_total = args.prof ? clock64() : 0;
            for (int gi = 0; gi < n_groups; gi++)
            for (int layer = 0; layer < n_layers; layer++) {
            const LayerView P = layer_view(layer);
            const int nkb = P.taps * P.kchunks;
            for (int slot = group_begin(gi); slot < group_begin(gi + 1); slot++, it++) {
                const int as = it & 1;
                const uint32_t aphase = (uint32_t)(it >> 1) & 1u;
                long long t0 = args.prof ? clock64() : 0;
                mbar_wait(tempty_bar(as), aphase ^ 1u);
                if (args.prof) pc_wait_tempty += clock64() - t0;
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(as * 256);
                if constexpr (CTA2) {
                    const int nd = P.taps == 9 ? 3 : 1;
                    uint32_t acc = 0;
                    for (int g = 0; g < P.kchunks * nd; g++) {
                        t0 = args.prof ? clock64() : 0;
                        mbar_wait(afull_bar(ra), rap);
                        if (args.prof) pc_wait_full += clock64() - t0;
                        for (int dyi = 0; dyi < nd; dyi++) {
                            t0 = args.prof ? clock64() : 0;
                            mbar_wait(bfull_bar(rb), rbp);
                            if (args.prof) pc_wait_full += clock64() - t0;
                            tc_fence_after();
                            // tap dy reads rows [16 (dy + 1), 16 (dy + 1) + 128) of the box: a 2 KB step, which keeps
                            // the 1024-byte swizzle atoms aligned
                            const uint64_t da = umma_desc_sw128(abox_addr(ra) + (uint32_t)((nd == 3 ? dyi : 1) * 2048));
                            const uint64_t db = umma_desc_sw128(btile_addr(rb));
                            if (elect_one()) {
#pragma unroll
                                for (int k = 0; k < TC_BK / 16; k++)
                                    tc2_mma<OT>(d_tmem, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, (acc | (uint32_t)k) != 0);
                                tc2_commit_mc(bempty_bar(rb));
                                if (dyi == nd - 1) tc2_commit_mc(aempty_bar(ra));
                            }
                            __syncwarp();
                            acc = 1;
                            if (++rb == NB) {
                                rb = 0;
                                rbp ^= 1u;
                            }
                        }
                        if (++ra == NA) {
                            ra = 0;
                            rap ^= 1u;
                        }
                    }
                    if (elect_one()) tc2_commit_mc(tfull_bar(as));
                    __syncwarp();
                    continue;
                }
                for (int kb = 0; kb < nkb; kb++) {
                    t0 = args.prof ? clock64() : 0;
                    mbar_wait(full_bar(stage), phase);
                    if (args.prof) pc_wait_full += clock64() - t0;
                    tc_fence_after();
                    const uint32_t a_addr = smem_base + stage * STAGE_BYTES;
                    const uint64_t da = umma_desc_sw128(a_addr);
                    const uint64_t db = umma_desc_sw128(a_addr + TC_A_BYTES);
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < TC_BK / 16; k++)  // +32 bytes per instruction (K = 16 x 2 B or 32 x 1 B) inside the 128-byte row
                            tc_mma<OT>(d_tmem, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc,
                                        (uint32_t)((kb | k) != 0));
                        tc_commit(empty_bar(stage));
                    }
                    __syncwarp();
                    if (++stage == NSTAGES) {
                        stage = 0;
                        phase ^= 1u;
                    }
                }
                if (elect_one()) tc_commit(tfull_bar(as));
                __syncwarp();
            }
            }
            if (args.prof && lane == 0) {
                args.prof[blockIdx.x * 16 + 1] = pc_wait_tempty;
                args.prof[blockIdx.x * 16 + 2] = pc_wait_full;
                args.prof[blockIdx.x * 16 + 3] = clock64() - pc_total;
                args.prof[blockIdx.x * 16 + 4] = it;
            }
        }
    } else if ((EPI == EPI_LN || EPI == EPI_LN_SE || EPI == EPI_LN73_GATHER || EPI == EPI_F32) || warp < 6) {
        const int quad = warp & 3;
        const int row = quad * 32 + lane;
        // pair kernels (shared activation box): accumulator row = (rank, board, file); orow = its row in memory
        const int orow = ((row >> 3) & 1) * 64 + (row >> 4) * 8 + (row & 7);
        const int te = (warp - 2) * 32 + lane;  // 0..255 (0..127 for the 4-warp epilogues)
        const int chalf = (warp - 2) >> 2;      // which 128-column half of the tile this warp owns
        int it = 0;
        long long pe_wait = 0, pe_work = 0, pe_stats = 0, pe_pool = 0, pe_fc = 0, pe_final = 0;
        const bool prof = args.prof != nullptr && te == 0;
        for (int gi = 0; gi < n_groups; gi++)
        for (int layer = 0; layer < n_layers; layer++) {
        const LayerView P = layer_view(layer);
        const bool is_se = P.se, se_fc = P.se_fc;
        if constexpr (TOWER) {
            // this layer's bias / LayerNorm parameters replace the previous layer's in shared memory
            epi_bar_sync();
            s_bias[te] = P.bias[te];
            s_gamma[te] = P.ln ? P.gamma[te] : 1.f;
            s_beta[te] = P.ln ? P.beta[te] : 0.f;
            if constexpr (OT::SCALED) s_scale[te] = P.scale[te];
            epi_bar_sync();
        }
        // end of a tile in the tower kernel: the tile's output (generic-proxy stores) is handed to the TMA
        // loads (async proxy) of the next layer through a per-tile mbarrier
        auto tile_done = [&](int sl) {
            if constexpr (TOWER) {
                asm volatile("fence.proxy.async;" ::: "memory");
                mbar_arrive(ready_bar(sl));
            }
        };
        for (int slot = group_begin(gi); slot < group_begin(gi + 1); slot++, it++) {
            const int work = work0 + slot * work_stride;
            const int tile = EPI == EPI_RAW ? work / args.n_splits : (CTA2 ? work * 2 + (int)cta_rank : work);
            const int split = EPI == EPI_RAW ? work % args.n_splits : 0;
            const int as = it & 1;
            const uint32_t aphase = (uint32_t)(it >> 1) & 1u;
            if (EPI == EPI_LN73_GATHER && as != (warp >= 6)) continue;  // the other warp set's tile
            long long tp0 = prof ? clock64() : 0;
            mbar_wait(tfull_bar(as), aphase);
            long long tp1 = prof ? clock64() : 0;
            pe_wait += tp1 - tp0;
            tc_fence_after();
            if (CTA2 && tile >= args.n_tiles) {
                // odd tile count: the second half of the last pair computes on zero-filled boards; nothing to store
                tc_fence_before();
                mbar_arrive_leader(tempty_bar(as));
                tile_done(slot);
                continue;
            }
            const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(as * 256);

            if constexpr (EPI == EPI_F32) {
                // ---- bias only: the fp32 accumulator goes to memory (this warp: 128 columns of its 32 rows) ----
                uint32_t r[32];
                const int c0 = chalf * 128;
                uint8_t *stg = s_stage + (warp - 2) * 2048;
                uint8_t *gtile = reinterpret_cast<uint8_t *>(static_cast<float *>(P.out) + (size_t)tile * TC_BM * BN + c0);
#pragma unroll 1
                for (int ch = 0; ch < 4; ch++) {
                    tmem_ld32(taddr + (uint32_t)(c0 + ch * 32), r);
#pragma unroll
                    for (int hf = 0; hf < 2; hf++) {
                        uint4 v[4];
#pragma unroll
                        for (int q = 0; q < 4; q++) {
                            float y[4];
#pragma unroll
                            for (int i = 0; i < 4; i++)
                                y[i] = __fadd_rn(__uint_as_float(r[hf * 16 + 4 * q + i]), s_bias[c0 + ch * 32 + hf * 16 + 4 * q + i]);
                            v[q] = make_uint4(__float_as_uint(y[0]), __float_as_uint(y[1]), __float_as_uint(y[2]), __float_as_uint(y[3]));
                        }
                        staged_store_64B_hbw(stg, lane, v, gtile + (ch * 32 + hf * 16) * 4, (size_t)BN * 4, quad);
                    }
                }
            } else if constexpr (EPI == EPI_RAW) {
                uint32_t r[32];
                uint8_t *stg = s_stage + (warp - 2) * 2048;
                const int wrow0 = tile * TC_BM + quad * 32;  // first global row of this warp
                uint8_t *gbase = reinterpret_cast<uint8_t *>(static_cast<float *>(args.out) +
                                                             ((size_t)split * args.m_rows + wrow0) * BN);
                const int rows_valid = args.m_rows - wrow0;
#pragma unroll 1
                for (int ch = 0; ch < BN / 32; ch++) {
                    tmem_ld32(taddr + ch * 32, r);
#pragma unroll
                    for (int hf = 0; hf < 2; hf++) {
                        uint4 v[4];
#pragma unroll
                        for (int q = 0; q < 4; q++)
                            v[q] = make_uint4(r[hf * 16 + 4 * q], r[hf * 16 + 4 * q + 1], r[hf * 16 + 4 * q + 2], r[hf * 16 + 4 * q + 3]);
                        staged_store_64B(stg, lane, v, gbase + (ch * 32 + hf * 16) * 4, (size_t)BN * 4, rows_valid);
                    }
                }
                if (args.vfin.counters) {
                    // ---- value head tail: the CTA that delivers the last split of this row tile finishes the tile.
                    //      Everybody's partial sums are made visible (fence), one thread counts the tile's arrivals. ----
                    const TcValueFinish &F = args.vfin;
                    __threadfence();
                    asm volatile("bar.sync 2, 128;" ::: "memory");
                    unsigned int *s_flag = reinterpret_cast<unsigned int *>(s_stat);
                    if (te == 0) {
                        const unsigned int old = atomicAdd(F.counters + tile, 1u);
                        const bool last = old == (unsigned int)args.n_splits - 1u;
                        if (last) F.counters[tile] = 0u;  // ready for the next launch
                        *s_flag = last ? 1u : 0u;
                    }
                    asm volatile("bar.sync 2, 128;" ::: "memory");
                    const bool last = *s_flag != 0u;
                    asm volatile("bar.sync 2, 128;" ::: "memory");  // the flag is read before the next work item overwrites it
                    if (last) {
                        // warp = rows quad, quad + 4, ... of the tile; lane = hidden units 4 lane .. 4 lane + 3 (one
                        // coalesced 512-byte row per load instruction, eight splits and four rows in flight)
                        __threadfence();
                        const float *pre = static_cast<const float *>(args.out);
                        const int nsp = args.n_splits;
                        float wm[SC_N_META][4], b1v[4], w2v[4], sv[4];
#pragma unroll
                        for (int i = 0; i < 4; i++) {
                            if constexpr (OT::SCALED) sv[i] = args.scale[4 * lane + i];
                            b1v[i] = F.b1[4 * lane + i];
                            w2v[i] = F.w2[4 * lane + i];
#pragma unroll
                            for (int k = 0; k < SC_N_META; k++) wm[k][i] = F.w_meta[k * BN + 4 * lane + i];
                        }
                        const float b2 = F.b2[0];
                        const int wq = warp - 2;  // 0..3
#pragma unroll 1
                        for (int r0 = wq; r0 < TC_BM; r0 += 16) {
                            float4 h[4];
                            int grow[4];
#pragma unroll
                            for (int u = 0; u < 4; u++) {
                                grow[u] = tile * TC_BM + r0 + 4 * u;
                                h[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                            }
                            // split order: a fixed fp32 sum; the loads of four splits are issued together (a split-at-a-time
                            // loop exposes one L2 latency per split: 16 x 0.35 us on the one-leaf path)
                            for (int sp0 = 0; sp0 < nsp; sp0 += 4) {
                                float4 p[4][4];
#pragma unroll
                                for (int d = 0; d < 4; d++)
#pragma unroll
                                    for (int u = 0; u < 4; u++)
                                        p[d][u] = (sp0 + d < nsp && grow[u] < args.m_rows)
                                                      ? __ldcg(reinterpret_cast<const float4 *>(pre + ((size_t)(sp0 + d) * args.m_rows + grow[u]) * BN) + lane)
                                                      : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                                for (int d = 0; d < 4; d++)
#pragma unroll
                                    for (int u = 0; u < 4; u++)
                                        if (sp0 + d < nsp) {  // (x + 0 is exact, but keep the operation count of the kernel form)
                                            h[u].x += p[d][u].x;
                                            h[u].y += p[d][u].y;
                                            h[u].z += p[d][u].z;
                                            h[u].w += p[d][u].w;
                                        }
                            }
#pragma unroll
                            for (int u = 0; u < 4; u++) {
                                if (grow[u] >= args.m_rows) continue;  // warp-uniform
                                const float *mt = F.meta + (size_t)grow[u] * 8;
                                float hv[4] = {h[u].x, h[u].y, h[u].z, h[u].w};
                                if constexpr (OT::SCALED)  // the hidden unit's weight scale, after the split sum (exact)
#pragma unroll
                                    for (int i = 0; i < 4; i++) hv[i] = __fmul_rn(hv[i], sv[i]);
                                float acc = 0.f;
#pragma unroll
                                for (int i = 0; i < 4; i++) {
#pragma unroll
                                    for (int k = 0; k < SC_N_META; k++) hv[i] = fmaf(wm[k][i], mt[k], hv[i]);
                                    acc = fmaf(w2v[i], fmaxf(hv[i] + b1v[i], 0.f), acc);
                                }
#pragma unroll
                                for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
                                if (lane == 0) F.value_out[grow[u]] = tanhf(acc + b2) * (mt[0] * 2.f - 1.f);
                            }
                        }
                    }
                }
            } else if constexpr (EPI == EPI_LN73_GATHER) {
                // ---- policy head: bias + LayerNorm(73), then the leaf's 64 x 73 policy map stays on the SM: rows
                //      0..63 of the tile are leaf 2*tile (warps of quadrants 0,1), rows 64..127 leaf 2*tile+1; thread =
                //      one square with its 73 channels in registers.  Even tiles are handled by epilogue warps 2..5, odd
                //      tiles by warps 6..9 (one accumulator stage and one shared-memory buffer each), so two tiles'
                //      epilogues run side by side. ----
                constexpr int LDL = 81;
                const int es = warp >= 6;
                float *s_logit = reinterpret_cast<float *>(s_y) + es * (Cfg::G_BYTES / 8);
                float *s_pri = s_logit + TC_BM * LDL;       // [2 leaves][SC_MAX_MOVES]
                float *s_red = s_pri + 2 * SC_MAX_MOVES;    // [4 quadrants][max, sum]
                float v[BN];
#pragma unroll
                for (int ch = 0; ch < BN / 16; ch++) {
                    uint32_t r[16];
                    tmem_ld16(taddr + ch * 16, r);
#pragma unroll
                    for (int j = 0; j < 16; j++) v[ch * 16 + j] = head_a(r[j], ch * 16 + j);
                }
                tc_fence_before();
                mbar_arrive(tempty_bar(as));  // the accumulator is free for the MMAs of tile it + 2
                float sum = 0.f;
#pragma unroll
                for (int c = 0; c < C_POLICY; c++) sum += v[c];
                float mean = sum * (1.f / C_POLICY);
                float sq = 0.f;
#pragma unroll
                for (int c = 0; c < C_POLICY; c++) {
                    const float d = v[c] - mean;
                    sq = fmaf(d, d, sq);
                }
                float rstd = rsqrtf(sq * (1.f / C_POLICY) + LN_EPS);
                if (!args.ln) {  // no normalisation (folded BatchNorm): gamma = 1, beta = 0 were loaded above
                    mean = 0.f;
                    rstd = 1.f;
                }
                float *mine = s_logit + row * LDL;
                float mx = -INFINITY;
#pragma unroll
                for (int c = 0; c < C_POLICY; c++) {
                    v[c] = (v[c] - mean) * rstd * s_gamma[c] + s_beta[c];
                    mine[c] = v[c];
                    mx = fmaxf(mx, v[c]);
                }
#pragma unroll
                for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
                if (lane == 0) s_red[quad * 2] = mx;
                gather_bar_sync(es);
                const int lf = quad >> 1;
                const float m = fmaxf(s_red[lf * 4], s_red[lf * 4 + 2]);
                float se = 0.f;
#pragma unroll
                for (int c = 0; c < C_POLICY; c++) se += __expf(v[c] - m);
#pragma unroll
                for (int o = 16; o; o >>= 1) se += __shfl_xor_sync(0xffffffffu, se, o);
                if (lane == 0) s_red[quad * 2 + 1] = se;
                gather_bar_sync(es);
                const float lsum = logf(s_red[lf * 4 + 1] + s_red[lf * 4 + 3]);
                const TcGather &G = args.gather;
                const int b = tile * 2 + lf;
                const int t64 = (quad & 1) * 32 + lane;
                int beg = 0, cnt = 0;
                if (b < G.n) {
                    beg = G.off ? G.off[b] : b * SC_MAX_MOVES;
                    cnt = G.off ? G.off[b + 1] - beg : G.cnt[b];
                    cnt = cnt > SC_MAX_MOVES ? SC_MAX_MOVES : cnt;
                    const int turn = G.pos[b].meta[0];
                    const float *L = s_logit + lf * 64 * LDL;
                    for (int k = t64; k < cnt; k += 64) {
                        const int idx = move_index_dev(G.moves[beg + k], turn, c_queen_dir, c_knight_type);
                        // flat NCHW index: channel idx / 64, square idx % 64 (py/module.py:75)
                        s_pri[lf * SC_MAX_MOVES + k] = idx >= 0 ? expf((L[(idx & 63) * LDL + (idx >> 6)] - m) - lsum) : 0.f;
                    }
                }
                gather_bar_sync(es);
                if (b < G.n) {
                    // `distr.iter().sum::<f32>() + 1e-5`: left-to-right f32 sum (chess.rs:891), every thread on its own
                    float tot = 0.f;
                    for (int k = 0; k < cnt; k++) tot += s_pri[lf * SC_MAX_MOVES + k];
                    tot += 1e-5f;
                    for (int k = t64; k < cnt; k += 64) G.priors[beg + k] = __fdiv_rn(s_pri[lf * SC_MAX_MOVES + k], tot);
                }
                gather_bar_sync(es);  // this warp set's next tile overwrites s_logit / s_pri
                continue;
            } else if constexpr (EPI == EPI_LN73) {
                uint32_t r[16];
                float sum = 0.f;
#pragma unroll 1
                for (int ch = 0; ch < BN / 16; ch++) {
                    tmem_ld16(taddr + ch * 16, r);
#pragma unroll
                    for (int j = 0; j < 16; j++)
                        if (ch * 16 + j < C_POLICY) sum += head_a(r[j], ch * 16 + j);
                }
                const float mean = args.ln ? sum * (1.f / C_POLICY) : 0.f;
                float sq = 0.f;
#pragma unroll 1
                for (int ch = 0; ch < BN / 16; ch++) {
                    tmem_ld16(taddr + ch * 16, r);
#pragma unroll
                    for (int j = 0; j < 16; j++)
                        if (ch * 16 + j < C_POLICY) {
                            float d = head_a(r[j], ch * 16 + j) - mean;
                            sq = fmaf(d, d, sq);
                        }
                }
                const float rstd = args.ln ? rsqrtf(sq * (1.f / C_POLICY) + LN_EPS) : 1.f;
                uint8_t *stg = s_stage + (warp - 2) * 2048;
                uint8_t *gbase = reinterpret_cast<uint8_t *>(static_cast<float *>(args.out) +
                                                             ((size_t)tile * TC_BM + quad * 32) * BN);
#pragma unroll 1
                for (int ch = 0; ch < BN / 16; ch++) {
                    tmem_ld16(taddr + ch * 16, r);
                    uint4 v[4];
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        float y[4];
#pragma unroll
                        for (int i = 0; i < 4; i++) {
                            const int c = ch * 16 + 4 * q + i;
                            y[i] = c < C_POLICY ? (head_a(r[4 * q + i], c) - mean) * rstd * s_gamma[c] + s_beta[c] : 0.f;
                        }
                        v[q] = make_uint4(__float_as_uint(y[0]), __float_as_uint(y[1]), __float_as_uint(y[2]), __float_as_uint(y[3]));
                    }
                    staged_store_64B(stg, lane, v, gbase + ch * 64, (size_t)BN * 4, 32);
                }
            } else {
                // ---- bias + LayerNorm(256) [+ SE + residual] ; this warp owns columns [c0, c0 + 128) of
                //      its 32 rows, the sibling warp (same TMEM quadrant) owns the other half --------------
                const int c0 = chalf * 128;
                const uint32_t tcol = taddr + (uint32_t)c0;
                uint32_t r[32];
                float mean, rstd;
                if (P.ln) {
                    // one TMEM pass: per 32-channel chunk the sum of a = acc + bias and its centred sum of squares,
                    // combined in the fixed tree of tc_ptx.cuh (the latency kernel computes the same chunks in other CTAs)
                    uint32_t r2[32];
                    float2 p0, p1, p2, p3;
                    auto chunk_pair = [&](int ch, float2 &pa, float2 &pb) {
                        tmem_ld32_nowait(tcol + ch * 32, r);
                        tmem_ld32_nowait(tcol + ch * 32 + 32, r2);
                        tmem_wait_ld();
                        float a0[32], a1[32];
#pragma unroll
                        for (int j = 0; j < 32; j++) {
                            a0[j] = acc_bias(r[j], c0 + ch * 32 + j);
                            a1[j] = acc_bias(r2[j], c0 + ch * 32 + 32 + j);
                        }
                        ln_chunk_stats(a0, pa.x, pa.y);
                        ln_chunk_stats(a1, pb.x, pb.y);
                    };
                    chunk_pair(0, p0, p1);
                    chunk_pair(2, p2, p3);
                    const float2 mine = ln_half(p0, p1, p2, p3);
                    *reinterpret_cast<float2 *>(s_stat + (chalf * 128 + row) * 2) = mine;
                    epi_bar_sync();
                    const float2 o = *reinterpret_cast<const float2 *>(s_stat + ((chalf ^ 1) * 128 + row) * 2);
                    ln_finish(chalf ? o : mine, chalf ? mine : o, LN_EPS, mean, rstd);
                } else {
                    // no normalisation (BatchNorm folded into weights and bias at export): y = acc + bias exactly
                    mean = 0.f;
                    rstd = 1.f;
                    epi_bar_sync();
                }
                long long tp2 = prof ? clock64() : 0;
                pe_stats += tp2 - tp1;
                uint8_t *stg = s_stage + (warp - 2) * 2048;
                // FC1 weights do not depend on anything computed here: request them before the pooling pass
                // so their L2 latency is hidden (thread = (hidden unit j, channel half hc))
                uint4 w1v[16];
                if (se_fc) {
                    const int j = te & 127, hc = te >> 7;
#pragma unroll
                    for (int u = 0; u < 8; u++) w1v[u] = __ldg(P.w1p + (hc * 16 + u) * 128 + j);
                }
                if (is_se) {
                    // ---- squeeze: per-board channel means of y = LN(conv) (fp32) -------------------
                    uint32_t rn[32];
                    tmem_ld32(tcol, r);
#pragma unroll
                    for (int ch = 0; ch < 4; ch++) {
                        // request the next 32 columns while this chunk is normalised and reduced
                        if (ch < 3) tmem_ld32_nowait(tcol + (ch + 1) * 32, (ch & 1) ? r : rn);
                        const uint32_t(&cur)[32] = (ch & 1) ? rn : r;
                        float y[32];
#pragma unroll
                        for (int j = 0; j < 32; j++) {
                            const int c = c0 + ch * 32 + j;
                            y[j] = ln_apply(acc_bias(cur[j], c), mean, rstd, s_gamma[c], s_beta[c]);
                        }
                        if constexpr (YSMEM) {
                            // keep LN(acc) in the operand type in shared memory: the final pass then needs neither
                            // TMEM nor the LayerNorm arithmetic again, and the accumulator can be handed back early
#pragma unroll
                            for (int q = 0; q < 4; q++) {
                                uint32_t pw[4];
#pragma unroll
                                for (int i = 0; i < 4; i++) pw[i] = OT::Park::pack2(y[8 * q + 2 * i], y[8 * q + 2 * i + 1]);
                                const int chunk = (c0 + ch * 32) / 8 + q;
                                *reinterpret_cast<uint4 *>(s_y + orow * 512 + ((chunk ^ (orow & 7)) << 4)) =
                                    make_uint4(pw[0], pw[1], pw[2], pw[3]);
                            }
                        }
                        if (se_fc) {  // (a residual-only block, use_se=False, has no pooling)
                            // partial sums per (quadrant, board) live in the (idle) store-staging area
                            int i0;
                            const float2 ps = warp_transpose_reduce_2boards(y, lane, i0);
                            float *s_poolx = reinterpret_cast<float *>(s_stage);
                            *reinterpret_cast<float2 *>(s_poolx + (quad * 2 + ((lane >> 3) & 1)) * 256 + c0 + ch * 32 + i0) = ps;
                        }
                        if (ch < 3) tmem_wait_ld();
                    }
                    if constexpr (YSMEM) {
                        tc_fence_before();
                        mbar_arrive_leader(tempty_bar(as));  // the accumulator is no longer needed
                    }
                    if (se_fc) {
                        // second half of the FC1 weights (the register file holds 10 warps at <= 168 registers,
                        // so only half of them could be requested before the pooling pass)
                        const int j = te & 127, hc = te >> 7;
#pragma unroll
                        for (int u = 8; u < 16; u++) w1v[u] = __ldg(P.w1p + (hc * 16 + u) * 128 + j);
                    }
                    epi_bar_sync();
                    if (prof) { const long long t = clock64(); pe_pool += t - tp2; tp2 = t; }
                    if (se_fc) {
#pragma unroll
                    for (int i = 0; i < 2; i++) {
                        const int idx = te + 256 * i;  // [board][channel]
                        const int b = idx >> 8, c = idx & 255;
                        const float *s_poolx = reinterpret_cast<const float *>(s_stage);
                        s_mean[idx] = ((s_poolx[b * 256 + c] + s_poolx[(2 + b) * 256 + c]) +
                                       (s_poolx[(4 + b) * 256 + c] + s_poolx[(6 + b) * 256 + c])) * (1.f / 64.f);
                    }
                    epi_bar_sync();
                    // ---- excitation FC1 (256 -> 128): thread = (hidden unit j, channel half hc), both boards
                    uint4 w2v[16];
                    {
                        const int j = te & 127, hc = te >> 7;
                        // four 32-channel chunk chains per board, then the fixed tree (tc_ptx.cuh)
                        auto chunk1 = [&](int k, float &a0, float &a1) {
                            a0 = 0.f;
                            a1 = 0.f;
#pragma unroll
                            for (int uu = 0; uu < 4; uu++) {
                                const int u = 4 * k + uu, q = hc * 16 + u;
                                float wf[8];
                                OT::unpack8(w1v[u], wf);
                                a0 = se_chain8(wf, *reinterpret_cast<const float4 *>(s_mean + q * 8),
                                               *reinterpret_cast<const float4 *>(s_mean + q * 8 + 4), a0);
                                a1 = se_chain8(wf, *reinterpret_cast<const float4 *>(s_mean + 256 + q * 8),
                                               *reinterpret_cast<const float4 *>(s_mean + 256 + q * 8 + 4), a1);
                            }
                        };
                        float xa0, xa1, xb0, xb1;
                        chunk1(0, xa0, xa1);
                        chunk1(1, xb0, xb1);
                        const float l0 = __fadd_rn(xa0, xb0), l1 = __fadd_rn(xa1, xb1);
                        chunk1(2, xa0, xa1);
                        chunk1(3, xb0, xb1);
                        // se_tree4: (p0 + p1) + (p2 + p3)
                        const float h0 = __fadd_rn(l0, __fadd_rn(xa0, xb0)), h1 = __fadd_rn(l1, __fadd_rn(xa1, xb1));
                        s_hidp[(hc * 2 + 0) * 128 + j] = h0;
                        s_hidp[(hc * 2 + 1) * 128 + j] = h1;
                    }
                    // FC2 weights (thread = channel te) are requested now and consumed two barriers later
#pragma unroll
                    for (int u = 0; u < 16; u++) w2v[u] = __ldg(P.w2p + u * 256 + te);
                    epi_bar_sync();
                    {
                        const int b = te >> 7, j = te & 127;  // [board][hidden unit]
                        s_hid[te] = se_hidden(P.b1[j], s_hidp[b * 128 + j], s_hidp[(2 + b) * 128 + j]);
                    }
                    epi_bar_sync();
                    // ---- FC2 (128 -> 256) + sigmoid: thread te owns channel te for both boards
                    {
                        auto chunk2 = [&](int k, float &a0, float &a1) {
                            a0 = 0.f;
                            a1 = 0.f;
#pragma unroll
                            for (int qq = 0; qq < 4; qq++) {
                                const int q = 4 * k + qq;
                                float wf[8];
                                OT::unpack8(w2v[q], wf);
                                a0 = se_chain8(wf, *reinterpret_cast<const float4 *>(s_hid + q * 8),
                                               *reinterpret_cast<const float4 *>(s_hid + q * 8 + 4), a0);
                                a1 = se_chain8(wf, *reinterpret_cast<const float4 *>(s_hid + 128 + q * 8),
                                               *reinterpret_cast<const float4 *>(s_hid + 128 + q * 8 + 4), a1);
                            }
                        };
                        float ya0, ya1, yb0, yb1;
                        chunk2(0, ya0, ya1);
                        chunk2(1, yb0, yb1);
                        const float m0 = __fadd_rn(ya0, yb0), m1 = __fadd_rn(ya1, yb1);
                        chunk2(2, ya0, ya1);
                        chunk2(3, yb0, yb1);
                        // se_fc2_sum: b2 + ((c0 + c1) + (c2 + c3))
                        const float g0 = __fadd_rn(P.b2[te], __fadd_rn(m0, __fadd_rn(ya0, yb0)));
                        const float g1 = __fadd_rn(P.b2[te], __fadd_rn(m1, __fadd_rn(ya1, yb1)));
                        s_gate[te] = se_sigmoid(g0);
                        s_gate[256 + te] = se_sigmoid(g1);
                    }
                    epi_bar_sync();
                    } else {
                        // residual-only block: gate = 1, so the final pass computes relu(y + x) exactly
                        s_gate[te] = 1.f;
                        s_gate[256 + te] = 1.f;
                        epi_bar_sync();
                    }
                    if (prof) { const long long t = clock64(); pe_fc += t - tp2; tp2 = t; }
                }

                if (YSMEM && is_se) {
                    // ---- final pass, elementwise and fully coalesced: thread te owns 16-byte chunk te % 32 of
                    //      rows te / 32 + 8 i; y from shared memory, x from global, out = relu(gate * y + x)
                    const int chunk = te & 31, r0 = te >> 5;
                    float g0[8], g1[8];
                    {
                        const float4 a0 = *reinterpret_cast<const float4 *>(s_gate + chunk * 8);
                        const float4 a1 = *reinterpret_cast<const float4 *>(s_gate + chunk * 8 + 4);
                        const float4 b0 = *reinterpret_cast<const float4 *>(s_gate + 256 + chunk * 8);
                        const float4 b1 = *reinterpret_cast<const float4 *>(s_gate + 256 + chunk * 8 + 4);
                        g0[0] = a0.x; g0[1] = a0.y; g0[2] = a0.z; g0[3] = a0.w; g0[4] = a1.x; g0[5] = a1.y; g0[6] = a1.z; g0[7] = a1.w;
                        g1[0] = b0.x; g1[1] = b0.y; g1[2] = b0.z; g1[3] = b0.w; g1[4] = b1.x; g1[5] = b1.y; g1[6] = b1.z; g1[7] = b1.w;
                    }
                    const size_t tile_row0 = (size_t)tile * TC_BM;
                    if constexpr (OT::BYTES == 2) {
                        const uint4 *xg = reinterpret_cast<const uint4 *>(P.resid + tile_row0 * BN) + chunk;
                        uint4 *og = reinterpret_cast<uint4 *>(static_cast<uint16_t *>(P.out) + tile_row0 * BN) + chunk;
#pragma unroll
                        for (int i0 = 0; i0 < 16; i0 += 8) {
                            uint4 xv[8];
#pragma unroll
                            for (int u = 0; u < 8; u++) xv[u] = xg[(size_t)(r0 + 8 * (i0 + u)) * (BN / 8)];
#pragma unroll
                            for (int u = 0; u < 8; u++) {
                                const int rr = r0 + 8 * (i0 + u);
                                const uint4 yv = *reinterpret_cast<const uint4 *>(s_y + rr * 512 + ((chunk ^ (rr & 7)) << 4));
                                const float *g = (i0 + u) < 8 ? g0 : g1;  // rows 0..63 are the tile's first board
                                const uint32_t yw[4] = {yv.x, yv.y, yv.z, yv.w};
                                const uint32_t xw[4] = {xv[u].x, xv[u].y, xv[u].z, xv[u].w};
                                uint32_t ow[4];
#pragma unroll
                                for (int k = 0; k < 4; k++) {
                                    const float o0 = fmaxf(fmaf(g[2 * k], OT::lo(yw[k]), OT::lo(xw[k])), 0.f);
                                    const float o1 = fmaxf(fmaf(g[2 * k + 1], OT::hi(yw[k]), OT::hi(xw[k])), 0.f);
                                    ow[k] = OT::pack2(o0, o1);
                                }
                                og[(size_t)rr * (BN / 8)] = make_uint4(ow[0], ow[1], ow[2], ow[3]);
                            }
                        }
                    } else {
                        // 1-byte operands: the chunk's 8 channels are 8 bytes of x and of the output; y is parked in
                        // OT::Park (bf16)
                        const uint2 *xg = reinterpret_cast<const uint2 *>(reinterpret_cast<const uint8_t *>(P.resid) + tile_row0 * BN) + chunk;
                        uint2 *og = reinterpret_cast<uint2 *>(static_cast<uint8_t *>(P.out) + tile_row0 * BN) + chunk;
#pragma unroll
                        for (int i0 = 0; i0 < 16; i0 += 8) {
                            uint2 xv[8];
#pragma unroll
                            for (int u = 0; u < 8; u++) xv[u] = xg[(size_t)(r0 + 8 * (i0 + u)) * (BN / 8)];
#pragma unroll
                            for (int u = 0; u < 8; u++) {
                                const int rr = r0 + 8 * (i0 + u);
                                const uint4 yv = *reinterpret_cast<const uint4 *>(s_y + rr * 512 + ((chunk ^ (rr & 7)) << 4));
                                const float *g = (i0 + u) < 8 ? g0 : g1;
                                const uint32_t yw[4] = {yv.x, yv.y, yv.z, yv.w};
                                float x[8], o[8];
                                OT::unpack4(xv[u].x, *reinterpret_cast<float(*)[4]>(x));
                                OT::unpack4(xv[u].y, *reinterpret_cast<float(*)[4]>(x + 4));
#pragma unroll
                                for (int k = 0; k < 4; k++) {
                                    o[2 * k] = fmaxf(fmaf(g[2 * k], OT::Park::lo(yw[k]), x[2 * k]), 0.f);
                                    o[2 * k + 1] = fmaxf(fmaf(g[2 * k + 1], OT::Park::hi(yw[k]), x[2 * k + 1]), 0.f);
                                }
                                og[(size_t)rr * (BN / 8)] = make_uint2(OT::pack4(o[0], o[1], o[2], o[3]), OT::pack4(o[4], o[5], o[6], o[7]));
                            }
                        }
                    }
                    if (prof) pe_final += clock64() - tp2;
                    tile_done(slot);
                    continue;  // the accumulator was released after the pooling pass
                }
                // ---- final pass of the LayerNorm-only layers: y (recomputed from TMEM), ReLU, store in the operand type --
                if constexpr (OT::BYTES == 1) {
                    // 1-byte operands: two 32-channel chunks make the lane's 64 bytes of the staged store
                    uint8_t *gtile = static_cast<uint8_t *>(P.out) + (size_t)tile * TC_BM * BN + c0;
                    uint32_t rm[32];
                    uint4 pk[4];
                    tmem_ld32(tcol, r);
#pragma unroll
                    for (int ch = 0; ch < 4; ch++) {
                        if (ch < 3) tmem_ld32_nowait(tcol + (ch + 1) * 32, (ch & 1) ? r : rm);
                        const uint32_t(&cur)[32] = (ch & 1) ? rm : r;
                        uint32_t w[8];
#pragma unroll
                        for (int j = 0; j < 8; j++) {
                            float y[4];
#pragma unroll
                            for (int i = 0; i < 4; i++) {
                                const int c = c0 + ch * 32 + 4 * j + i;
                                y[i] = ln_apply(acc_bias(cur[4 * j + i], c), mean, rstd, s_gamma[c], s_beta[c]);
                                if (P.relu) y[i] = fmaxf(y[i], 0.f);
                            }
                            w[j] = OT::pack4(y[0], y[1], y[2], y[3]);
                        }
                        pk[(ch & 1) * 2] = make_uint4(w[0], w[1], w[2], w[3]);
                        pk[(ch & 1) * 2 + 1] = make_uint4(w[4], w[5], w[6], w[7]);
                        if (ch & 1) staged_store_64B_hbw(stg, lane, pk, gtile + (ch - 1) * 32, (size_t)BN, quad);
                        if (ch < 3) tmem_wait_ld();
                    }
                } else {
                    uint8_t *gtile = reinterpret_cast<uint8_t *>(static_cast<uint16_t *>(P.out) + (size_t)tile * TC_BM * BN + c0);
                    uint32_t rm[32];
                    tmem_ld32(tcol, r);
#pragma unroll
                    for (int ch = 0; ch < 4; ch++) {
                        if (ch < 3) tmem_ld32_nowait(tcol + (ch + 1) * 32, (ch & 1) ? r : rm);
                        const uint32_t(&cur)[32] = (ch & 1) ? rm : r;
                        uint4 pk[4];
#pragma unroll
                        for (int j = 0; j < 16; j++) {
                            const int c = c0 + ch * 32 + 2 * j;
                            float y0 = ln_apply(__fadd_rn(__uint_as_float(cur[2 * j]), s_bias[c]), mean, rstd, s_gamma[c], s_beta[c]);
                            float y1 = ln_apply(__fadd_rn(__uint_as_float(cur[2 * j + 1]), s_bias[c + 1]), mean, rstd, s_gamma[c + 1],
                                                s_beta[c + 1]);
                            if (P.relu) {
                                y0 = fmaxf(y0, 0.f);
                                y1 = fmaxf(y1, 0.f);
                            }
                            const uint32_t hv = OT::pack2(y0, y1);
                            if ((j & 3) == 0) pk[j >> 2].x = hv;
                            else if ((j & 3) == 1) pk[j >> 2].y = hv;
                            else if ((j & 3) == 2) pk[j >> 2].z = hv;
                            else pk[j >> 2].w = hv;
                        }
                        staged_store_64B_hbw(stg, lane, pk, gtile + ch * 64, (size_t)BN * 2, quad);
                        if (ch < 3) tmem_wait_ld();
                    }
                }
                if (prof) pe_final += clock64() - tp2;
            }
            tc_fence_before();
            if (CTA2) mbar_arrive_leader(tempty_bar(as));
            else mbar_arrive(tempty_bar(as));
            tile_done(slot);
            if (prof) pe_work += clock64() - tp1;
        }
        }
        if (prof) {
            args.prof[blockIdx.x * 16 + 5] = pe_wait;
            args.prof[blockIdx.x * 16 + 6] = pe_work;
            args.prof[blockIdx.x * 16 + 7] = pe_stats;
            args.prof[blockIdx.x * 16 + 8] = pe_pool;
            args.prof[blockIdx.x * 16 + 9] = pe_fc;
            args.prof[blockIdx.x * 16 + 10] = pe_final;
        }
    }

    tc_fence_before();
    __syncthreads();
    if (CTA2) cluster_sync_all();  // neither CTA may leave while the pair's MMAs / remote arrives can touch it
    if (warp == 1) {
        tc_fence_after();
        if (CTA2)
            asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
        else
            asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// ---- host side ------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode()
{
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

struct ActMap {
    const void *ptr;
    int rows, c;
    CUtensorMap map;
};

// bn == 256: a convolution of the CTA-pair kernels, whose weight box {64, 128} is the half of the weight rows one CTA of
// the pair stages; otherwise a single-CTA head GEMM with the weight box {64, bn}
struct TcConv {
    CUtensorMap map_w;
    int taps, k_per_tap, bn, epi;
    TcOp op = TC_OP_BF16;                  // operand type
    const float *scale = nullptr;          // TC_OP_E4M3: per-output-channel weight scales
    int split_pairs = 0, split_kreal = 0;  // FP32 parity mode: (A plane, B plane) pairs of the bf16x3 split
    uint8_t split_ap[8] = {0}, split_bp[8] = {0};
    const float *bias, *gamma, *beta;
    const uint4 *se_w1p = nullptr, *se_w2p = nullptr;
    const float *se_b1 = nullptr, *se_b2 = nullptr;
    std::vector<ActMap> act_maps;
};

int tc_encode_map(CUtensorMap *m, CUtensorMapDataType dt, const void *ptr, int rank, const cuuint64_t *dims,
                  const cuuint64_t *strides, const cuuint32_t *box, const char *what, bool swizzle128)
{
    EncodeTiledFn enc = get_encode();
    if (!enc) {
        set_error("cuTensorMapEncodeTiled not available from the driver");
        return SC_E_CUDA;
    }
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(m, dt, (cuuint32_t)rank, const_cast<void *>(ptr), dims, strides, box,
                     estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error(std::string("cuTensorMapEncodeTiled(") + what + ") failed: " + std::to_string((int)r));
        return SC_E_CUDA;
    }
    return SC_OK;
}

// bytes per element of a tensor-map type, and the channels of one 128-byte K chunk
static cuuint64_t tmap_bytes(CUtensorMapDataType dt) { return dt == CU_TENSOR_MAP_DATA_TYPE_UINT8 ? 1 : 2; }
static cuuint32_t tmap_bk(CUtensorMapDataType dt) { return (cuuint32_t)(128 / tmap_bytes(dt)); }

// activations as a 4-D tensor {C, file, rank, board}, box = one K chunk of channels of two whole boards
static int make_act_map_4d(CUtensorMapDataType dt, const void *ptr, int boards, int c, CUtensorMap *m)
{
    const cuuint64_t eb = tmap_bytes(dt);
    cuuint64_t dims[4] = {(cuuint64_t)c, 8, 8, (cuuint64_t)boards};
    cuuint64_t strides[3] = {(cuuint64_t)c * eb, (cuuint64_t)c * 8 * eb, (cuuint64_t)c * 64 * eb};
    cuuint32_t box[4] = {tmap_bk(dt), 8, 8, 2};
    return tc_encode_map(m, dt, ptr, 4, dims, strides, box, "activations 4d");
}

// the same activations as {C, file, board, rank}: a box of 64 channels x 8 files x 2 boards x 10 ranks lands in
// shared memory with rows ordered (rank, board, file), so the three dy taps are 2 KB apart in ONE box
int tc_make_act_map_hbw(CUtensorMapDataType dt, const void *ptr, int boards, int c, CUtensorMap *m)
{
    const cuuint64_t eb = tmap_bytes(dt);
    cuuint64_t dims[4] = {(cuuint64_t)c, 8, (cuuint64_t)boards, 8};
    cuuint64_t strides[3] = {(cuuint64_t)c * eb, (cuuint64_t)c * 64 * eb, (cuuint64_t)c * 8 * eb};
    cuuint32_t box[4] = {tmap_bk(dt), 8, 2, 10};
    return tc_encode_map(m, dt, ptr, 4, dims, strides, box, "activations (rank, board, file)");
}

// plain row-major [rows][k] matrix, box = one K chunk x 128 rows
static int make_act_map_2d(CUtensorMapDataType dt, const void *ptr, int rows, int k, CUtensorMap *m)
{
    cuuint64_t dims[2] = {(cuuint64_t)k, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)k * tmap_bytes(dt)};
    cuuint32_t box[2] = {tmap_bk(dt), TC_BM};
    return tc_encode_map(m, dt, ptr, 2, dims, strides, box, "activations 2d");
}

template <int BN, int EPI, bool A4D, class OT> static int set_smem_attr()
{
    SCB_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<BN, EPI, A4D, false, false, OT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  TcCfg<BN>::SMEM_BYTES));
    return SC_OK;
}

// the dynamic shared-memory sizes of the non-split kernels of one operand type
template <class OT> static int set_conv_attrs()
{
    SCB_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<256, EPI_LN, true, true, false, OT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  TcCfg<256, true>::SMEM_BYTES));
    SCB_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<256, EPI_LN_SE, true, true, false, OT>,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<256, true, true>::SMEM_BYTES));
    SCB_CHECK((set_smem_attr<LD_POLICY, EPI_LN73, true, OT>()));
    SCB_CHECK((set_smem_attr<LD_POLICY, EPI_LN73_GATHER, true, OT>()));
    SCB_CHECK((set_smem_attr<N_VALUE_HIDDEN, EPI_RAW, false, OT>()));
    return SC_OK;
}

static CUtensorMapDataType tmap_type(TcOp op)
{
    return op == TC_OP_E4M3 ? OpE4m3::TMAP : op == TC_OP_FP16 ? OpFp16::TMAP : OpBf16::TMAP;
}

int tc_conv_create(TcConv **out, const __nv_bfloat16 *w, int taps, int k_per_tap, int bn, int epi, const float *bias,
                   const float *gamma, const float *beta, TcOp op, const float *scale)
{
    if ((op == TC_OP_E4M3) != (scale != nullptr) || k_per_tap % tc_op_bk(op) != 0) {
        set_error("tc_conv_create: e4m3 weights need their scales (and only they), K a whole number of chunks");
        return SC_E_INVAL;
    }
    TcConv *c = new TcConv();
    c->op = op;
    c->scale = scale;
    c->taps = taps;
    c->k_per_tap = k_per_tap;
    c->bn = bn;
    c->epi = epi;
    c->bias = bias;
    c->gamma = gamma;
    c->beta = beta;
    // weights [taps * bn rows][k_per_tap], K-major
    const CUtensorMapDataType dt = tmap_type(op);
    cuuint64_t dims[2] = {(cuuint64_t)k_per_tap, (cuuint64_t)taps * bn};
    cuuint64_t strides[1] = {(cuuint64_t)k_per_tap * tmap_bytes(dt)};
    cuuint32_t box[2] = {tmap_bk(dt), (cuuint32_t)(bn == 256 ? bn / 2 : bn)};
    int rc = tc_encode_map(&c->map_w, dt, w, 2, dims, strides, box, "weights");
    if (rc != SC_OK) {
        delete c;
        return rc;
    }
    // function attributes belong to the device (context): set them once per device, not once per process
    static std::mutex attr_mu;
    static std::map<std::pair<int, int>, bool> attr_done;
    int dev = 0;
    SCB_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(attr_mu);
    bool &attr_set = attr_done[{dev, (int)op}];
    if (!attr_set) {
        SCB_CHECK(op == TC_OP_E4M3 ? set_conv_attrs<OpE4m3>() : op == TC_OP_FP16 ? set_conv_attrs<OpFp16>() : set_conv_attrs<OpBf16>());
        attr_set = true;
    }
    *out = c;
    return SC_OK;
}

// FP32 parity mode: a 3x3 / 1x1 convolution to 256 channels as a bf16x3 split GEMM with fp32 output (EPI_F32).
// w3: bf16 [taps][256][3 * cin_pad], the weights' three bf16 planes side by side along K; the activations come as
// bf16 [boards][64][a_planes * cin_pad] (a_planes = 3, or 1 for inputs that are exact in bf16: the 0/1 input planes).
// Terms kept: a_i * b_j with i + j <= 2 (error ~2^-24 relative, i.e. fp32 level), smallest first.
int tc_split_conv_create(TcConv **out, const __nv_bfloat16 *w3, int taps, int cin_pad, int a_planes, const float *bias)
{
    if (a_planes != 1 && a_planes != 3) {
        set_error("tc_split_conv_create: a_planes must be 1 or 3");
        return SC_E_INVAL;
    }
    TcConv *c = new TcConv();
    c->taps = taps;
    c->k_per_tap = a_planes * cin_pad;  // channels of the activation tensor
    c->bn = 256;
    c->epi = EPI_F32;
    c->bias = bias;
    c->gamma = nullptr;
    c->beta = nullptr;
    cuuint64_t dims[2] = {(cuuint64_t)3 * cin_pad, (cuuint64_t)taps * 256};
    cuuint64_t strides[1] = {(cuuint64_t)3 * cin_pad * 2};
    cuuint32_t box2[2] = {TC_BK, 128};
    int rc = tc_encode_map(&c->map_w, OpBf16::TMAP, w3, 2, dims, strides, box2, "split weights (pair half)");
    if (rc != SC_OK) {
        delete c;
        return rc;
    }
    c->split_kreal = cin_pad / TC_BK;
    if (a_planes == 3) {
        static const uint8_t ap[6] = {0, 1, 2, 0, 1, 0}, bp[6] = {2, 1, 0, 1, 0, 0};
        c->split_pairs = 6;
        memcpy(c->split_ap, ap, 6);
        memcpy(c->split_bp, bp, 6);
    } else {
        static const uint8_t bp[3] = {2, 1, 0};
        c->split_pairs = 3;
        memcpy(c->split_bp, bp, 3);
    }
    int dev = 0;
    SCB_CUDA(cudaGetDevice(&dev));
    (void)dev;
    SCB_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<256, EPI_F32, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  TcCfg<256, true>::SMEM_BYTES));
    *out = c;
    return SC_OK;
}

void tc_conv_set_se(TcConv *c, const void *w1p, const float *b1, const void *w2p, const float *b2)
{
    c->se_w1p = static_cast<const uint4 *>(w1p);
    c->se_w2p = static_cast<const uint4 *>(w2p);
    c->se_b1 = b1;
    c->se_b2 = b2;
}

void tc_conv_destroy(TcConv *c) { delete c; }


// SCB200_PHASE_PROFILE=1: [grid][16] phase cycle counters, one buffer per device, sized from the device's SM count
static int prof_buffer(int num_sms, cudaStream_t st, long long **out)
{
    static std::mutex mu;
    static std::map<int, std::pair<long long *, int>> bufs;
    int dev = 0;
    SCB_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(mu);
    auto &b = bufs[dev];
    if (b.second < num_sms) {
        if (b.first) cudaFree(b.first);
        b.first = nullptr;
        SCB_CUDA(cudaMalloc(&b.first, (size_t)num_sms * 16 * sizeof(long long)));
        b.second = num_sms;
    }
    SCB_CUDA(cudaMemsetAsync(b.first, 0, (size_t)num_sms * 16 * sizeof(long long), st));
    *out = b.first;
    return SC_OK;
}

// ---- whole-tower kernel --------------------------------------------------------------------------------
struct TcTower {
    TowerLayer *d_layers = nullptr;
    int n_layers = 0;
    TcOp op = TC_OP_BF16;
};

int tc_tower_create(TcTower **out, const TcTowerLayerDesc *descs, int n, int boards_alloc, TcOp op)
{
    std::vector<TowerLayer> h((size_t)n);
    for (int i = 0; i < n; i++) {
        const TcConv *c = descs[i].conv;
        if (!c || c->bn != 256 || (c->epi != EPI_LN && c->epi != EPI_LN_SE)) {
            set_error("tc_tower_create: layer is not a 256-wide tower convolution");
            return SC_E_INVAL;
        }
        if (c->op != op) {
            set_error("tc_tower_create: layer of another operand type");
            return SC_E_INVAL;
        }
        memset(&h[i], 0, sizeof(TowerLayer));
        SCB_CHECK(tc_make_act_map_hbw(tmap_type(op), descs[i].in, boards_alloc, c->k_per_tap, &h[i].map_a));
        h[i].map_w = c->map_w;
        h[i].out = descs[i].out;
        h[i].resid = descs[i].resid;
        h[i].bias = c->bias;
        h[i].gamma = c->gamma;
        h[i].beta = c->beta;
        h[i].se_w1p = c->se_w1p;
        h[i].se_w2p = c->se_w2p;
        h[i].se_b1 = c->se_b1;
        h[i].se_b2 = c->se_b2;
        h[i].taps = c->taps;
        h[i].kchunks = c->k_per_tap / tc_op_bk(op);
        h[i].scale = c->scale;
        h[i].relu = descs[i].relu;
        // se: 1 = squeeze-excitation gate, 2 = residual + ReLU only (`use_se=False`, no SE weights)
        h[i].se = c->epi == EPI_LN_SE ? (c->se_w1p ? 1 : 2) : 0;
        h[i].ln = c->gamma != nullptr;  // no LayerNorm parameters: BatchNorm folded into weights + bias at export
        if (h[i].se && !descs[i].resid) {
            set_error("tc_tower_create: residual layer without block input");
            return SC_E_INVAL;
        }
    }
    TcTower *t = new TcTower();
    t->n_layers = n;
    t->op = op;
    if (cudaMalloc(&t->d_layers, sizeof(TowerLayer) * (size_t)n) != cudaSuccess ||
        cudaMemcpy(t->d_layers, h.data(), sizeof(TowerLayer) * (size_t)n, cudaMemcpyHostToDevice) != cudaSuccess) {
        delete t;
        set_error("tc_tower_create: device allocation failed");
        return SC_E_CUDA;
    }
    if (op == TC_OP_E4M3)
        SCB_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<256, EPI_LN_SE, true, true, true, OpE4m3>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<256, true, true>::SMEM_BYTES));
    else if (op == TC_OP_FP16)
        SCB_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<256, EPI_LN_SE, true, true, true, OpFp16>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<256, true, true>::SMEM_BYTES));
    else
        SCB_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<256, EPI_LN_SE, true, true, true>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<256, true, true>::SMEM_BYTES));
    *out = t;
    return SC_OK;
}

void tc_tower_destroy(TcTower *t)
{
    if (!t) return;
    cudaFree(t->d_layers);
    delete t;
}

// returns SC_E_STATE (without an error message) when the batch needs more tile slots per CTA than the
// kernel tracks; the caller then runs the layers one launch at a time
int tc_tower_launch(TcTower *t, int n_boards, int num_sms, int group, cudaStream_t st, int max_layers)
{
    if (n_boards <= 0) return SC_OK;
    const int n_tiles = (n_boards + 1) / 2;
    const int n_pairs = (n_tiles + 1) / 2;
    int g2 = 2 * n_pairs;
    if (g2 > (num_sms & ~1)) g2 = num_sms & ~1;
    const int slots = (n_pairs + g2 / 2 - 1) / (g2 / 2);
    if (slots > TC_MAX_SLOTS) return SC_E_STATE;
    TcArgs a;
    memset(&a, 0, sizeof(a));
    a.n_tiles = n_tiles;
    a.n_splits = 1;
    a.layers = t->d_layers;
    a.n_layers = max_layers > 0 && max_layers < t->n_layers ? max_layers : t->n_layers;
    a.group = group;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(g2);
    cfg.blockDim = dim3(TC_THREADS);
    cfg.dynamicSmemBytes = TcCfg<256, true, true>::SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    static CUtensorMap dummy;  // the layer array carries the tensor maps
    long long *d_prof = nullptr;
    static const bool want_prof = getenv("SCB200_PHASE_PROFILE") != nullptr;
    if (want_prof) {
        SCB_CHECK(prof_buffer(num_sms, st, &d_prof));
        a.prof = d_prof;
    }
    if (t->op == TC_OP_E4M3)
        SCB_CUDA(cudaLaunchKernelEx(&cfg, tc_gemm_kernel<256, EPI_LN_SE, true, true, true, OpE4m3>, dummy, dummy, a));
    else if (t->op == TC_OP_FP16)
        SCB_CUDA(cudaLaunchKernelEx(&cfg, tc_gemm_kernel<256, EPI_LN_SE, true, true, true, OpFp16>, dummy, dummy, a));
    else
        SCB_CUDA(cudaLaunchKernelEx(&cfg, tc_gemm_kernel<256, EPI_LN_SE, true, true, true>, dummy, dummy, a));
    SCB_CUDA(cudaGetLastError());
    if (want_prof) {
        std::vector<long long> h((size_t)num_sms * 16);
        SCB_CUDA(cudaStreamSynchronize(st));
        SCB_CUDA(cudaMemcpy(h.data(), d_prof, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
        double acc[16] = {0};
        for (int b = 0; b < g2; b += 2)  // leader CTAs carry the MMA counters
            for (int k = 0; k < 16; k++) acc[k] += (double)h[b * 16 + k] / (g2 / 2);
        fprintf(stderr,
                "[tower layers=%d grid=%d] tiles/cta %.2f | producer wait_empty %.0f | mma: total %.0f wait_tmem_empty %.0f "
                "wait_full %.0f | epilogue: wait_tmem_full %.0f work %.0f (stats %.0f pool %.0f fc %.0f final %.0f)\n",
                t->n_layers, g2, acc[4], acc[0], acc[3], acc[1], acc[2], acc[5], acc[6], acc[7], acc[8], acc[9], acc[10]);
    }
    return SC_OK;
}

// the launch of one convolution / head GEMM with operand type OT (a: everything but the pair / gather / finish choice)
template <class OT>
static int conv_launch_kernel(const TcConv *c, const CUtensorMap &ma, TcArgs &a, int grid, int num_sms, cudaStream_t st,
                              const __nv_bfloat16 *resid, const TcGather *gather, const TcValueFinish *finish)
{
    const bool pair = c->bn == 256;
    if (pair) {
        const int n_pairs = (a.n_tiles + 1) / 2;
        int g2 = 2 * n_pairs;
        if (g2 > (num_sms & ~1)) g2 = num_sms & ~1;
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(g2);
        cfg.blockDim = dim3(TC_THREADS);
        cfg.dynamicSmemBytes = c->epi == EPI_LN_SE ? TcCfg<256, true, true>::SMEM_BYTES : TcCfg<256, true>::SMEM_BYTES;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        if (c->epi == EPI_F32) {
            if constexpr (std::is_same<OT, OpBf16>::value) {
                SCB_CUDA(cudaLaunchKernelEx(&cfg, tc_gemm_kernel<256, EPI_F32, true, true>, ma, c->map_w, a));
            } else {
                set_error("tc_conv_launch: the split fp32 epilogue has bf16 operands only");
                return SC_E_INVAL;
            }
        } else if (c->epi == EPI_LN)
            SCB_CUDA(cudaLaunchKernelEx(&cfg, tc_gemm_kernel<256, EPI_LN, true, true, false, OT>, ma, c->map_w, a));
        else {
            if (!resid) {
                set_error("tc_conv_launch: residual epilogue without block input");
                return SC_E_INVAL;
            }
            SCB_CUDA(cudaLaunchKernelEx(&cfg, tc_gemm_kernel<256, EPI_LN_SE, true, true, false, OT>, ma, c->map_w, a));
        }
    } else {
        switch (c->epi) {
        case EPI_LN73:
            if (gather) {
                a.gather = *gather;
                tc_gemm_kernel<LD_POLICY, EPI_LN73_GATHER, true, false, false, OT><<<grid, TC_THREADS, TcCfg<LD_POLICY>::SMEM_BYTES, st>>>(ma, c->map_w, a);
            } else
                tc_gemm_kernel<LD_POLICY, EPI_LN73, true, false, false, OT><<<grid, TC_THREADS, TcCfg<LD_POLICY>::SMEM_BYTES, st>>>(ma, c->map_w, a);
            break;
        case EPI_RAW:
            if (finish) a.vfin = *finish;
            tc_gemm_kernel<N_VALUE_HIDDEN, EPI_RAW, false, false, false, OT><<<grid, TC_THREADS, TcCfg<N_VALUE_HIDDEN>::SMEM_BYTES, st>>>(
                ma, c->map_w, a);
            break;
        default:
            set_error("tc_conv_launch: bad epilogue");
            return SC_E_INVAL;
        }
    }
    return SC_OK;
}

int tc_conv_launch(TcConv *c, const __nv_bfloat16 *in, int rows_alloc, int n_units, void *out,
                   const __nv_bfloat16 *resid, int relu, int n_splits, int num_sms, cudaStream_t st, const TcGather *gather,
                   const TcValueFinish *finish)
{
    if (n_units <= 0) return SC_OK;
    const bool a4d = c->epi != EPI_RAW;
    // CTA-pair (cta_group::2) kernels for every 256-wide convolution: clusters of two CTAs, each pair owns a 256-row
    // tile (4 boards) -- also for a single tile: the arithmetic must not depend on the batch size
    const bool pair = c->bn == 256;
    const CUtensorMap *ma = nullptr;
    for (auto &m : c->act_maps)
        if (m.ptr == in && m.rows == rows_alloc && m.c == c->k_per_tap) ma = &m.map;
    if (!ma) {
        ActMap am;
        am.ptr = in;
        am.rows = rows_alloc;
        am.c = c->k_per_tap;
        // (the split kernel of the FP32 parity mode is created with the bf16 operand type)
        const CUtensorMapDataType dt = tmap_type(c->op);
        if (pair)
            SCB_CHECK(tc_make_act_map_hbw(dt, in, rows_alloc, c->k_per_tap, &am.map));
        else if (a4d)
            SCB_CHECK(make_act_map_4d(dt, in, rows_alloc, c->k_per_tap, &am.map));
        else
            SCB_CHECK(make_act_map_2d(dt, in, rows_alloc, c->k_per_tap, &am.map));
        c->act_maps.push_back(am);
        ma = &c->act_maps.back().map;
    }
    TcArgs a;
    memset(&a, 0, sizeof(a));
    long long *d_prof = nullptr;
    static const bool want_prof = getenv("SCB200_PHASE_PROFILE") != nullptr;
    if (want_prof) {
        SCB_CHECK(prof_buffer(num_sms, st, &d_prof));
        a.prof = d_prof;
    }
    a.out = out;
    a.resid = resid;
    a.bias = c->bias;
    a.gamma = c->gamma;
    a.beta = c->beta;
    a.se_w1p = c->se_w1p;
    a.se_w2p = c->se_w2p;
    a.se_b1 = c->se_b1;
    a.se_b2 = c->se_b2;
    a.relu = relu;
    a.ln = c->gamma != nullptr;
    a.scale = c->scale;
    a.n_splits = n_splits > 0 ? n_splits : 1;
    a.m_rows = n_units;
    if (a4d) {
        a.n_tiles = (n_units + 1) / 2;  // units = boards, two per tile
        a.taps = c->taps;
        a.kchunks = c->k_per_tap / tc_op_bk(c->op);
        if (c->split_pairs > 0) {
            a.split_pairs = c->split_pairs;
            a.split_kreal = c->split_kreal;
            memcpy(a.split_ap, c->split_ap, 8);
            memcpy(a.split_bp, c->split_bp, 8);
            a.kchunks = c->split_pairs * c->split_kreal;
        }
    } else {
        a.n_tiles = (n_units + TC_BM - 1) / TC_BM;  // units = rows
        a.taps = 1;
        a.kchunks = c->k_per_tap / tc_op_bk(c->op) / a.n_splits;
    }
    const int n_work = a4d ? a.n_tiles : a.n_tiles * a.n_splits;
    const int grid = n_work < num_sms ? n_work : num_sms;
    if (c->op == TC_OP_E4M3)
        SCB_CHECK(conv_launch_kernel<OpE4m3>(c, *ma, a, grid, num_sms, st, resid, gather, finish));
    else if (c->op == TC_OP_FP16)
        SCB_CHECK(conv_launch_kernel<OpFp16>(c, *ma, a, grid, num_sms, st, resid, gather, finish));
    else
        SCB_CHECK(conv_launch_kernel<OpBf16>(c, *ma, a, grid, num_sms, st, resid, gather, finish));
    SCB_CUDA(cudaGetLastError());
    if (want_prof) {
        // debugging aid: per-phase SM-cycle counters of this launch, averaged over CTAs (synchronous!)
        std::vector<long long> h((size_t)num_sms * 16);
        SCB_CUDA(cudaStreamSynchronize(st));
        SCB_CUDA(cudaMemcpy(h.data(), d_prof, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
        double acc[16] = {0};
        for (int b = 0; b < grid; b++)
            for (int k = 0; k < 16; k++) acc[k] += (double)h[b * 16 + k] / grid;
        fprintf(stderr,
                "[tc epi=%d taps=%d grid=%d] tiles/cta %.2f | producer wait_empty %.0f | mma: total %.0f wait_tmem_empty %.0f "
                "wait_full %.0f | epilogue: wait_tmem_full %.0f work %.0f (stats %.0f pool %.0f fc %.0f final %.0f)\n",
                c->epi, c->taps, grid, acc[4], acc[0], acc[3], acc[1], acc[2], acc[5], acc[6], acc[7], acc[8], acc[9], acc[10]);
    }
    return SC_OK;
}

}  // namespace scb
