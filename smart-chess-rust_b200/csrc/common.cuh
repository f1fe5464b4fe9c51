// Shared declarations for the B200 leaf-evaluation backend (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <string>

#include "../../include/sc_b200.h"

namespace scb {

void set_error(const std::string &msg);

#define SCB_CUDA(expr)                                                                         \
    do {                                                                                       \
        cudaError_t e__ = (expr);                                                              \
        if (e__ != cudaSuccess) {                                                              \
            scb::set_error(std::string(#expr) + ": " + cudaGetErrorString(e__));               \
            return SC_E_CUDA;                                                                  \
        }                                                                                      \
    } while (0)

#define SCB_CHECK(expr)                                                                        \
    do {                                                                                       \
        int r__ = (expr);                                                                      \
        if (r__ != SC_OK) return r__;                                                          \
    } while (0)

constexpr int C_TOWER = 256;     // tower width (py/module.py:120)
constexpr int C_IN = 112;        // input planes
constexpr int C_IN_PAD = 128;    // tensor-core modes: planes padded to two 16-bit K chunks (one e4m3 chunk)
constexpr int C_SE = 128;        // SqueezeExcitation(256, 128) (py/module.py:29-33)
constexpr int C_POLICY = 73;
constexpr int LD_POLICY = 80;    // row stride of the policy logits buffer [B][64][80]
constexpr int N_VALUE_HIDDEN = 128;
constexpr float LN_EPS = 1e-6f;  // timm LayerNorm2d

// ---- encode.cu ---------------------------------------------------------------------------
// planes: one warp per position. out element (b, s, c), s = rank*8+file, c < ld.
int launch_encode_i8(const sc_position *d_pos, int n, int8_t *out, int32_t *meta_out, cudaStream_t st);
int launch_encode_f32(const sc_position *d_pos, int n, float *out /*[n][64][112]*/, float *meta_out /*[n][8]*/,
                      cudaStream_t st);
int launch_encode_bf16(const sc_position *d_pos, int n, __nv_bfloat16 *out /*[n][64][128]*/,
                       float *meta_out /*[n][8]*/, cudaStream_t st);
int launch_encode_fp16(const sc_position *d_pos, int n, __half *out /*[n][64][128]*/, float *meta_out /*[n][8]*/,
                       cudaStream_t st);
int launch_encode_e4m3(const sc_position *d_pos, int n, uint8_t *out /*[n][64][128]*/, float *meta_out /*[n][8]*/,
                       cudaStream_t st);
// NCHW float planes (sc_forward_only input) -> NHWC
int launch_nchw_to_nhwc_f32(const float *in, int n, float *out, cudaStream_t st);
int launch_nchw_to_nhwc_bf16(const float *in, int n, __nv_bfloat16 *out, cudaStream_t st);
int launch_nchw_to_nhwc_fp16(const float *in, int n, __half *out, cudaStream_t st);
int launch_nchw_to_nhwc_e4m3(const float *in, int n, uint8_t *out, cudaStream_t st);

// ---- policy.cu ----------------------------------------------------------------------------
// logits [n][64][LD_POLICY] fp32 (square-major) -> per-leaf log-sum-exp, legal-move gather,
// exp, sequential renormalisation; optional move index dump / full logp dump.
int launch_move_index(const sc_position *d_pos, const sc_move *d_moves, const int32_t *d_off, int n,
                      int32_t *d_index, cudaStream_t st);
// moves are CSR (d_off[n+1], d_cnt == nullptr) or strided (d_off == nullptr: leaf b owns
// [b*SC_MAX_MOVES, +d_cnt[b]) of d_moves and d_priors)
int launch_policy_gather(const float *logits, const sc_position *d_pos, const sc_move *d_moves,
                         const int32_t *d_off, const int32_t *d_cnt, int n, float *d_priors, cudaStream_t st);
// visit counts -> training target: dist[b][move_index(m_k)] = cnt_k / (sum_k cnt_k + 1e-5) (src/lib.rs:104-112)
int launch_dist_scatter(const sc_position *d_pos, const sc_move *d_moves, const uint32_t *d_counts,
                        const int32_t *d_off, int n, float *d_dist /*[n][4672]*/, cudaStream_t st);
int launch_policy_logp_full(const float *logits, int n, float *d_logp /*[n][4672]*/, cudaStream_t st);

// ---- movegen.cu ---------------------------------------------------------------------------
// the attack tables of host/chess_rules.hpp to the device (once per engine, before the first launch)
int upload_move_tables(cudaStream_t st);
// one thread per leaf: the legal moves of pos[i] (en-passant square d_ep[i], or -1 for all when d_ep == nullptr) in
// python-chess order into d_moves[i * SC_MAX_MOVES ..], their number into d_cnt[i], and into d_term[i] 0, a
// termination code of chess_rules.hpp (T_CHECKMATE / T_STALEMATE) when there is none, or PREDICT_OVERFLOW when the
// position has more than SC_MAX_MOVES pseudo-legal moves (then at most SC_MAX_MOVES are written)
constexpr int PREDICT_OVERFLOW = -1;
int launch_legal_moves(const sc_position *d_pos, const int8_t *d_ep, int n, sc_move *d_moves, int32_t *d_cnt,
                       int32_t *d_term, cudaStream_t st);
// the replay's statuses: 0, or REPLAY_STATUS(ply, reason) for the first move it rejects, ply counted from the game start
enum { REPLAY_NOT_OURS = 1, REPLAY_BAD_TARGET, REPLAY_BAD_PROMO, REPLAY_NO_PROMO };
__host__ __device__ constexpr int32_t REPLAY_STATUS(int ply, int reason) { return ply << 3 | reason; }
size_t replay_scratch_bytes(int64_t positions);
// sc_set_roots, one thread per root: replays root r's moves d_stack[d_off[r], d_off[r+1]) from the initial position and
// keeps its records (replay_scratch_bytes(d_off[n] + n) bytes of d_rec in all), its final position in d_root_pos[r] and
// its status in d_status[r]
namespace chess { struct Position; }
int launch_root_replay(const sc_move *d_stack, const int32_t *d_off, int n, void *d_rec, chess::Position *d_root_pos,
                       int32_t *d_status, cudaStream_t st);
// an evaluator's slot table: slot g's records at d_rec + replay_scratch_bytes(g * (SC_MAX_STACK + 1)), its final
// position in d_slot_pos[g] and its plies in d_slot_plies[g].  One thread per update u: replays d_stack[d_off[u],
// d_off[u+1]) into slot d_slot[u], from the initial position or (d_append[u] != 0) from the slot's stored position,
// appending to its records; the status into d_status[u].  The caller keeps the plies within SC_MAX_STACK
int launch_slot_replay(const sc_move *d_stack, const int32_t *d_off, const int32_t *d_slot, const int8_t *d_append,
                       int n, void *d_rec, chess::Position *d_slot_pos, int32_t *d_slot_plies, int32_t *d_status,
                       cudaStream_t st);
// sc_predict_stack / sc_predict_path / an evaluator's leaves, one thread per leaf: leaf i starts from root d_root[i] of
// the sc_set_roots table above (d_root_off = the d_off it was built from), or of a slot table when d_slot_plies is
// given (d_root_rec / d_root_pos: its records and positions), or from the initial position when d_root == nullptr (no
// table is then read), replays d_path[d_off[i], d_off[i+1]) and packs the game as host::pack_position does with d_n_hist[i]
// history slots (nullptr: min(SC_LOOKBACK, plies + 1)) into d_pos[i], its python-chess ep_square into d_ep[i], and its
// status into d_status[i] (after a rejected move the leaf is packed from the moves before it).  d_scratch:
// replay_scratch_bytes(d_off[n] + n) bytes, the path's records
int launch_path_replay(const void *d_root_rec, const int32_t *d_root_off, const int32_t *d_slot_plies,
                       const chess::Position *d_root_pos, const int32_t *d_root, const sc_move *d_path,
                       const int32_t *d_off, const int8_t *d_n_hist, int n, void *d_scratch, sc_position *d_pos,
                       int8_t *d_ep, int32_t *d_status, cudaStream_t st);

// ---- tower_f32.cu -------------------------------------------------------------------------
// C[M][N] = gather_taps(A)[M][TAPS*K] * W[TAPS*K][ldw] + bias ; A is [rows][lda] fp32
// n_splits > 1 (taps == 1, no bias): split-K over gridDim.z, partial sums to out[split][M][ldo]
int launch_gemm_f32(int taps, const float *A, int lda, const float *W, int ldw, const float *bias, float *out,
                    int ldo, int M, int N, int K, cudaStream_t st, int n_splits = 1);
// planes (optional): the result also as three bf16 planes [rows][3 * C] (hi | mid | lo), the operand format of the
// tensor-core FP32 parity mode
int launch_ln_f32(float *x, int rows, int C, int ld, const float *gamma, const float *beta, int relu,
                  cudaStream_t st, __nv_bfloat16 *planes = nullptr);
int launch_se_res_f32(const float *y, const float *x, float *out, int n, const float *w1t, const float *b1,
                      const float *w2t, const float *b2, cudaStream_t st, __nv_bfloat16 *planes = nullptr);
// scale (fp8 mode): the hidden units' weight scales, applied to the split sum
int launch_value_finish(const float *hidden_pre, int n_split, int n, const float *meta, const float *w_meta,
                        const float *b1, const float *w2, const float *b2, float *value_out, cudaStream_t st,
                        const float *scale = nullptr);

// ---- tower_bf16.cu (tcgen05) --------------------------------------------------------------
// The tensor-core modes share these kernels and interfaces.  The operand type selects fp16 or e4m3 operands instead of
// bf16, and then every operand buffer below (weights, activations; typed __nv_bfloat16) holds fp16 bit patterns, or
// e4m3 bytes ([..][k] with k one byte each).  e4m3 weights come with `scale`: per output channel a power of two that the
// epilogue multiplies the accumulator by.
enum TcOp { TC_OP_BF16 = 0, TC_OP_FP16 = 1, TC_OP_E4M3 = 2 };
// channels per K chunk (one 128-byte swizzle row): 64 16-bit or 128 8-bit elements
constexpr int tc_op_bk(TcOp op) { return op == TC_OP_E4M3 ? 128 : 64; }
struct TcConv;  // opaque per-layer state (tensor maps)
enum { TC_EPI_LN = 0, TC_EPI_LN_SE = 1, TC_EPI_LN73 = 2, TC_EPI_RAW = 3 };
// w: bf16 [taps][bn][k_per_tap] (K-major B operand); bn = 256 (tower / head 1x1 convs),
// 80 (policy 256->73, rows 73..79 zero) or 128 (value FC, taps = 1, k_per_tap = 16384)
int tc_conv_create(TcConv **out, const __nv_bfloat16 *w, int taps, int k_per_tap, int bn, int epi, const float *bias,
                   const float *gamma, const float *beta, TcOp op, const float *scale = nullptr);
// FP32 parity mode: conv to 256 channels as a bf16x3 split GEMM on the tensor cores, fp32 [boards * 64][256] out (+ bias).
// w3 = bf16 [taps][256][3 * cin_pad] (three planes side by side along K), activations bf16 [boards][64][a_planes * cin_pad]
int tc_split_conv_create(TcConv **out, const __nv_bfloat16 *w3, int taps, int cin_pad, int a_planes, const float *bias);
// squeeze-excitation weights for TC_EPI_LN_SE: fc1 packed [32][128][8], fc2 packed [16][256][8], in the operand type
void tc_conv_set_se(TcConv *c, const void *w1p, const float *b1, const void *w2p, const float *b2);
void tc_conv_destroy(TcConv *c);
// convs: in = bf16 NHWC [rows_alloc boards][64][k_per_tap], n_units = boards.
// value FC (TC_EPI_RAW): in = bf16 [rows_alloc][16384], n_units = rows, out = fp32 [n_splits][n_units][128].
// TC_EPI_LN73 with `gather`: the policy map stays on the SM; log-softmax, legal-move gather and renormalisation
// (policy.cu's policy_gather_kernel) run in the epilogue and only the priors are written.
struct TcGather {
    const sc_position *pos;  // [n] (side to move)
    const sc_move *moves;    // CSR by off, or strided by SC_MAX_MOVES with cnt when off == nullptr
    const int32_t *off, *cnt;
    float *priors;           // same layout as moves
    int n;
};
// TC_EPI_RAW with `finish`: the value head's tail (tower_f32.cu's value_finish_kernel) runs inside the split-K GEMM --
// the CTA that delivers the LAST of a row tile's split-K partial sums adds them up in split order, adds the meta columns
// and the bias, ReLU, FC 128 -> 1, tanh, white-perspective flip, and writes the values (py/module.py:95-106, 147-149).
struct TcValueFinish {
    const float *meta;     // [n][8]
    const float *w_meta;   // [7][128]
    const float *b1, *w2, *b2;
    float *value_out;      // [n]
    unsigned int *counters;  // one per 128-row tile, zero between launches (the finishing CTA resets its tile's)
};
int tc_conv_launch(TcConv *c, const __nv_bfloat16 *in, int rows_alloc, int n_units, void *out,
                   const __nv_bfloat16 *resid, int relu, int n_splits, int num_sms, cudaStream_t st,
                   const TcGather *gather = nullptr, const TcValueFinish *finish = nullptr);

// whole-tower kernel: every 256-wide convolution of the residual tower in ONE launch (layers in order)
struct TcTower;
struct TcTowerLayerDesc {
    TcConv *conv;
    const __nv_bfloat16 *in;     // bf16 NHWC [boards_alloc][64][conv k_per_tap]
    void *out;                   // bf16 NHWC [boards_alloc][64][256]
    const __nv_bfloat16 *resid;  // SE layers: block input (may alias out)
    int relu;
};
int tc_tower_create(TcTower **out, const TcTowerLayerDesc *descs, int n, int boards_alloc, TcOp op);
// group = tiles per CTA carried through all layers together (0 = all of the CTA's tiles)
// max_layers > 0: only the first max_layers layers (sc_debug_tower's layer-by-layer comparison)
int tc_tower_launch(TcTower *t, int n_boards, int num_sms, int group, cudaStream_t st, int max_layers = 0);
void tc_tower_destroy(TcTower *t);

// ---- tower_lat.cu: latency path for small batches (one 2-board tile per cluster of 8 / 4 CTAs) ------------------
struct LatTower;
struct LatLayerDesc {
    const __nv_bfloat16 *w;      // [taps][256][cin_pad] (the throughput kernel's B operand)
    int taps, cin_pad;
    const __nv_bfloat16 *in;     // bf16 NHWC [boards_alloc][64][cin_pad]
    void *out;                   // bf16 NHWC [boards_alloc][64][256]
    const __nv_bfloat16 *resid;  // residual layers: block input (may alias out)
    const float *bias, *gamma, *beta;
    int relu, ln;
    int se;                      // 0: LN (+ReLU); 1: LN + squeeze-excitation + residual + ReLU; 2: LN + residual + ReLU
    // SE weights sliced per cluster rank: fc1 [CL][32][128 / CL] x 8 bf16, fc2 [CL][16][256 / CL] x 8 bf16
    const void *se_w1s8, *se_w2s8, *se_w1s4, *se_w2s4;
    const float *se_b1, *se_b2;
};
int lat_tower_create(LatTower **out, const LatLayerDesc *descs, int n, int boards_alloc, bool fp16);
// largest batch the latency kernel takes (one wave of clusters); 0 if it cannot run on this device
int lat_tower_max_boards(const LatTower *t);
// SC_E_STATE (no message) when the batch does not fit: run the throughput kernel instead
int lat_tower_launch(LatTower *t, int n_boards, cudaStream_t st, int max_layers = 0);
void lat_tower_destroy(LatTower *t);

}  // namespace scb
