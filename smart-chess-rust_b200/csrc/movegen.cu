// Legal moves of every leaf on the device, for sc_predict (the `state.legal_moves()` half of `Game::predict`,
// src/game.rs:3-15, src/backends/torch.rs:96-106).
//
// One thread per leaf runs host/chess_rules.hpp's generator -- the same code as the host driver, so python-chess's
// generation order is defined in one place -- and writes each legal move straight into the leaf's strided output slot
// (leaf i owns moves[i * SC_MAX_MOVES, +SC_MAX_MOVES), the layout sc_eval_submit's gather reads).  The attack tables
// (70 KB) live in global memory: too large for constant memory, and the lookups diverge across threads.
#include "common.cuh"
#include "host/chess_rules.hpp"

namespace scb {
namespace chess {

static __device__ Tables g_tables;

__device__ const Tables &device_tables() { return g_tables; }

}  // namespace chess

namespace {

// writes the legal moves of one leaf into its slot; never past SC_MAX_MOVES
struct SlotSink {
    sc_move *out;
    int n;
    __device__ void add(int f, int t, int p)
    {
        if (n < SC_MAX_MOVES) out[n] = sc_move{(uint8_t)f, (uint8_t)t, (uint8_t)p, 0};
        n++;
    }
};

}  // namespace

constexpr int MOVEGEN_THREADS = 64;

__global__ void __launch_bounds__(MOVEGEN_THREADS) legal_moves_kernel(const sc_position *__restrict__ pos,
                                                                      const int8_t *__restrict__ ep_square, int n,
                                                                      sc_move *__restrict__ moves,
                                                                      int32_t *__restrict__ move_cnt,
                                                                      int32_t *__restrict__ term)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    chess::Position p;
    p.set_packed(pos[i], ep_square ? ep_square[i] : -1);
    SlotSink sink{moves + (size_t)i * SC_MAX_MOVES, 0};
    const int seen = p.gen_legal(sink);
    const int cnt = sink.n < SC_MAX_MOVES ? sink.n : SC_MAX_MOVES;
    move_cnt[i] = cnt;
    int code = chess::T_NONE;
    if (seen > SC_MAX_MOVES)
        code = PREDICT_OVERFLOW;  // not a legal position (a legal one has at most 218 moves): the call fails
    else if (cnt == 0)
        code = p.in_check() ? chess::T_CHECKMATE : chess::T_STALEMATE;
    term[i] = code;
}

int upload_move_tables(cudaStream_t st)
{
    SCB_CUDA(cudaMemcpyToSymbolAsync(chess::g_tables, &chess::host_tables(), sizeof(chess::Tables), 0,
                                     cudaMemcpyHostToDevice, st));
    return SC_OK;
}

int launch_legal_moves(const sc_position *d_pos, const int8_t *d_ep, int n, sc_move *d_moves, int32_t *d_cnt,
                       int32_t *d_term, cudaStream_t st)
{
    if (n <= 0) return SC_OK;
    legal_moves_kernel<<<(n + MOVEGEN_THREADS - 1) / MOVEGEN_THREADS, MOVEGEN_THREADS, 0, st>>>(d_pos, d_ep, n, d_moves,
                                                                                               d_cnt, d_term);
    SCB_CUDA(cudaGetLastError());
    return SC_OK;
}

}  // namespace scb
