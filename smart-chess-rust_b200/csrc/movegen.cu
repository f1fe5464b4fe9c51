// Legal moves of every leaf on the device, for sc_predict (the `state.legal_moves()` half of `Game::predict`,
// src/game.rs:3-15, src/backends/torch.rs:96-106), and the replay that packs each leaf from its move stack for
// sc_predict_stack.
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

// ---- sc_predict_stack: replay and pack ------------------------------------------------------------------------------
// Serial per leaf: each ply depends on the last.  What the repetition walk needs of every replayed position goes to a
// global scratch rather than a per-thread array (local memory is reserved for every resident thread), and
// chess::is_repetition walks it exactly as the host Game walks its stack.

namespace {

// one replayed position: its transposition key and halfmove clock, and whether the move played from it is irreversible
struct ReplayPly {
    chess::TKey key;
    int32_t halfmove, irreversible;
};

// chess::is_repetition's history over one leaf's replay: ply[k] = the position after k moves
struct ReplayHistory {
    const ReplayPly *ply;
    __device__ chess::u64 occupancy(int k) const { return ply[k].key.w | ply[k].key.b; }
    __device__ chess::TKey key(int k) const { return ply[k].key; }
    __device__ bool irreversible(int k) const { return ply[k].irreversible != 0; }
};

// the replay's checks (Board.push verifies no legality either; from/to < 64 and promo are checked on the host)
__device__ int replay_reject(const chess::Position &p, const sc_move &m)
{
    using namespace chess;
    const u64 from = bit(m.from), to = bit(m.to);
    if (!(p.occ[p.turn] & from)) return REPLAY_NOT_OURS;
    if ((p.occ[p.turn] | p.pt[KING]) & to) return REPLAY_BAD_TARGET;
    const bool last_rank = (p.pt[PAWN] & from) && rank_of(m.to) == (p.turn == WHITE ? 7 : 0);
    if (m.promo && !last_rank) return REPLAY_BAD_PROMO;
    if (!m.promo && last_rank) return REPLAY_NO_PROMO;
    return 0;
}

}  // namespace

constexpr int REPLAY_THREADS = 32;

__global__ void __launch_bounds__(REPLAY_THREADS) replay_kernel(const sc_move *__restrict__ stack,
                                                                const int32_t *__restrict__ off,
                                                                const int8_t *__restrict__ n_hist, int n,
                                                                ReplayPly *__restrict__ scratch,
                                                                sc_position *__restrict__ pos, int8_t *__restrict__ ep,
                                                                int32_t *__restrict__ status)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int base = off[i];
    const sc_move *mv = stack + base;
    ReplayPly *h = scratch + base + i;  // plies + 1 positions per leaf
    int len = off[i + 1] - base, st = 0;
    chess::Position p;
    p.set_start();
    for (int k = 0;; k++) {
        const chess::TKey key = chess::tkey(p);
        h[k].key = key;
        h[k].halfmove = p.halfmove;
        if (k == len) break;
        const sc_move m = mv[k];
        const int why = replay_reject(p, m);
        if (why) {
            st = REPLAY_STATUS(k, why);
            len = k;
            break;
        }
        const chess::Move cm{m.from, m.to, m.promo};
        // Position::is_irreversible, with its has_legal_ep() read off the key (key.ep is the ep square only if legal)
        h[k].irreversible = p.is_zeroing(cm) || p.reduces_castling(cm) || key.ep >= 0;
        p.push(cm);
    }
    int nh = n_hist ? n_hist[i] : SC_LOOKBACK;
    if (nh > len + 1) nh = len + 1;
    sc_position &o = pos[i];
    chess::pack_meta(p, o.meta);
    o.n_hist = nh;
    ep[i] = (int8_t)p.ep;
    status[i] = st;
    const ReplayHistory rh{h};
    for (int s = 0; s < SC_LOOKBACK; s++) {
        if (s < nh) {
            const int ply = len - s, hm = h[ply].halfmove;
            uint64_t rep = 0;
            if (chess::is_repetition(rh, ply, hm, 2)) rep = 1 | (chess::is_repetition(rh, ply, hm, 3) ? 2 : 0);
            chess::pack_slot(h[ply].key.pt, h[ply].key.w, rep, o.slot[s]);
        } else {
            for (int j = 0; j < 8; j++) o.slot[s][j] = 0;
        }
    }
}

size_t replay_scratch_bytes(int64_t positions) { return sizeof(ReplayPly) * (size_t)positions; }

int launch_replay(const sc_move *d_stack, const int32_t *d_off, const int8_t *d_n_hist, int n, void *d_scratch,
                  sc_position *d_pos, int8_t *d_ep, int32_t *d_status, cudaStream_t st)
{
    if (n <= 0) return SC_OK;
    replay_kernel<<<(n + REPLAY_THREADS - 1) / REPLAY_THREADS, REPLAY_THREADS, 0, st>>>(
        d_stack, d_off, d_n_hist, n, static_cast<ReplayPly *>(d_scratch), d_pos, d_ep, d_status);
    SCB_CUDA(cudaGetLastError());
    return SC_OK;
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
