// Legal moves of every leaf on the device, for sc_predict (the `state.legal_moves()` half of `Game::predict`,
// src/game.rs:3-15, src/backends/torch.rs:96-106), and the replay that packs each leaf from its move stack for
// sc_predict_stack, or from a stored root and its path for sc_set_roots / sc_predict_path and an evaluator's slots.
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

// ---- sc_predict_stack / sc_set_roots / sc_predict_path: replay and pack ---------------------------------------------
// Serial per leaf: each ply depends on the last.  What the repetition walk needs of every replayed position goes to a
// global scratch rather than a per-thread array (local memory is reserved for every resident thread), and
// chess::is_repetition walks it exactly as the host Game walks its stack.  sc_set_roots keeps these records of each
// root game in a persistent table; sc_predict_path continues a stored root's final position with the leaf's path and
// walks the root's records, then the path's.

namespace {

// one replayed position: its transposition key and halfmove clock, and whether the move played from it is irreversible
struct ReplayPly {
    chess::TKey key;
    int32_t halfmove, irreversible;
};

// chess::is_repetition's history over replay records; Records::at(k) = the record of the position after k moves
template <class Records> struct PlyHistory : Records {
    __device__ chess::u64 occupancy(int k) const { return this->at(k).key.w | this->at(k).key.b; }
    __device__ chess::TKey key(int k) const { return this->at(k).key; }
    __device__ bool irreversible(int k) const { return this->at(k).irreversible != 0; }
};

// a stored root of `root_plies` moves, then the leaf's path: the root's records up to its last move, the path's
// (path[0] = the root's final position, recorded again by the path replay) from there on.  A path from the initial
// position has root_plies = 0 and reads path[] alone
struct RootPathRecords {
    const ReplayPly *root, *path;
    int root_plies;
    __device__ const ReplayPly &at(int k) const { return k < root_plies ? root[k] : path[k - root_plies]; }
};
using PathHistory = PlyHistory<RootPathRecords>;

// where path_replay_kernel finds the records and the plies of root r.  sc_set_roots' table: root r's records at
// off[r] + r, off[r + 1] - off[r] plies
struct OffsetRoots {
    const int32_t *off;
    __device__ int64_t base(int r) const { return off[r] + r; }
    __device__ int plies(int r) const { return off[r + 1] - off[r]; }
};
// an evaluator's slot table: slot r's records at r * (SC_MAX_STACK + 1), n[r] plies
struct SlotRoots {
    const int32_t *n;
    __device__ int64_t base(int r) const { return (int64_t)r * (SC_MAX_STACK + 1); }
    __device__ int plies(int r) const { return n[r]; }
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

// plays mv[0, len) on p, ply by ply: the record h[k] of the position before move k (h[len]: the final position), the
// move's checks, then Position::push.  A rejected move k ends the replay with len = k and returns
// REPLAY_STATUS(ply0 + k, why) (ply0: the plies played before p); 0 when every move is played
__device__ __forceinline__ int replay_moves(chess::Position &p, const sc_move *mv, int &len, ReplayPly *h, int ply0)
{
    for (int k = 0;; k++) {
        const chess::TKey key = chess::tkey(p);
        h[k].key = key;
        h[k].halfmove = p.halfmove;
        if (k == len) return 0;
        const sc_move m = mv[k];
        const int why = replay_reject(p, m);
        if (why) {
            len = k;
            return REPLAY_STATUS(ply0 + k, why);
        }
        const chess::Move cm{m.from, m.to, m.promo};
        // Position::is_irreversible, with its has_legal_ep() read off the key (key.ep is the ep square only if legal)
        h[k].irreversible = p.is_zeroing(cm) || p.reduces_castling(cm) || key.ep >= 0;
        p.push(cm);
    }
}

// host::pack_position of the position p reached after `plies` moves, with min(nh, plies + 1) history slots read off h
template <class History>
__device__ __forceinline__ void pack_replayed(const History &h, const chess::Position &p, int plies, int nh,
                                              sc_position &o)
{
    if (nh > plies + 1) nh = plies + 1;
    chess::pack_meta(p, o.meta);
    o.n_hist = nh;
    for (int s = 0; s < SC_LOOKBACK; s++) {
        if (s < nh) {
            const int ply = plies - s, hm = h.at(ply).halfmove;
            uint64_t rep = 0;
            if (chess::is_repetition(h, ply, hm, 2)) rep = 1 | (chess::is_repetition(h, ply, hm, 3) ? 2 : 0);
            chess::pack_slot(h.at(ply).key.pt, h.at(ply).key.w, rep, o.slot[s]);
        } else {
            for (int j = 0; j < 8; j++) o.slot[s][j] = 0;
        }
    }
}

}  // namespace

constexpr int REPLAY_THREADS = 32;

// sc_set_roots, one thread per root: root r's records (plies + 1) at rec + off[r] + r, its final position and status
__global__ void __launch_bounds__(REPLAY_THREADS) root_replay_kernel(const sc_move *__restrict__ stack,
                                                                     const int32_t *__restrict__ off, int n,
                                                                     ReplayPly *__restrict__ rec,
                                                                     chess::Position *__restrict__ root_pos,
                                                                     int32_t *__restrict__ status)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const int base = off[r];
    int len = off[r + 1] - base;
    chess::Position p;
    p.set_start();
    status[r] = replay_moves(p, stack + base, len, rec + base + r, 0);
    root_pos[r] = p;
}

// an evaluator's root updates, one thread per updated slot: update u replays stack[off[u], off[u+1]) into slot slot[u],
// from the initial position or (append[u]) from the slot's stored position after its n_plies[slot] moves, and keeps
// the records from that ply on, the final position, the plies and status[u]
__global__ void __launch_bounds__(REPLAY_THREADS) slot_replay_kernel(const sc_move *__restrict__ stack,
                                                                     const int32_t *__restrict__ off,
                                                                     const int32_t *__restrict__ slot,
                                                                     const int8_t *__restrict__ append, int n,
                                                                     ReplayPly *__restrict__ rec,
                                                                     chess::Position *__restrict__ slot_pos,
                                                                     int32_t *__restrict__ n_plies,
                                                                     int32_t *__restrict__ status)
{
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= n) return;
    const int g = slot[u], base = off[u];
    int len = off[u + 1] - base, ply0 = 0;
    chess::Position p;
    if (append[u]) {
        p = slot_pos[g];
        ply0 = n_plies[g];
    } else {
        p.set_start();
    }
    status[u] = replay_moves(p, stack + base, len, rec + SlotRoots{}.base(g) + ply0, ply0);
    slot_pos[g] = p;
    n_plies[g] = ply0 + len;
}

// sc_predict_stack / sc_predict_path / an evaluator's leaves, one thread per leaf: root[i]'s stored position (root ==
// nullptr: the initial position) continued with path[off[i], off[i+1]) (records in the per-call scratch), packed over
// the root's records and the path's
template <class Roots>
__global__ void __launch_bounds__(REPLAY_THREADS) path_replay_kernel(
    const ReplayPly *__restrict__ root_rec, Roots roots,
    const chess::Position *__restrict__ root_pos, const int32_t *__restrict__ root, const sc_move *__restrict__ path,
    const int32_t *__restrict__ off, const int8_t *__restrict__ n_hist, int n, ReplayPly *__restrict__ scratch,
    sc_position *__restrict__ pos, int8_t *__restrict__ ep, int32_t *__restrict__ status)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int base = off[i];
    ReplayPly *h = scratch + base + i;  // plies + 1 positions per leaf
    int len = off[i + 1] - base;
    chess::Position p;
    const ReplayPly *rh = nullptr;
    int root_plies = 0;
    if (root) {
        const int r = root[i];
        root_plies = roots.plies(r);
        rh = root_rec + roots.base(r);
        p = root_pos[r];
    } else {
        p.set_start();
    }
    status[i] = replay_moves(p, path + base, len, h, root_plies);
    ep[i] = (int8_t)p.ep;
    const PathHistory ph{{rh, h, root_plies}};
    pack_replayed(ph, p, root_plies + len, n_hist ? n_hist[i] : SC_LOOKBACK, pos[i]);
}

size_t replay_scratch_bytes(int64_t positions) { return sizeof(ReplayPly) * (size_t)positions; }

int launch_root_replay(const sc_move *d_stack, const int32_t *d_off, int n, void *d_rec, chess::Position *d_root_pos,
                       int32_t *d_status, cudaStream_t st)
{
    if (n <= 0) return SC_OK;
    root_replay_kernel<<<(n + REPLAY_THREADS - 1) / REPLAY_THREADS, REPLAY_THREADS, 0, st>>>(
        d_stack, d_off, n, static_cast<ReplayPly *>(d_rec), d_root_pos, d_status);
    SCB_CUDA(cudaGetLastError());
    return SC_OK;
}

int launch_slot_replay(const sc_move *d_stack, const int32_t *d_off, const int32_t *d_slot, const int8_t *d_append,
                       int n, void *d_rec, chess::Position *d_slot_pos, int32_t *d_slot_plies, int32_t *d_status,
                       cudaStream_t st)
{
    if (n <= 0) return SC_OK;
    slot_replay_kernel<<<(n + REPLAY_THREADS - 1) / REPLAY_THREADS, REPLAY_THREADS, 0, st>>>(
        d_stack, d_off, d_slot, d_append, n, static_cast<ReplayPly *>(d_rec), d_slot_pos, d_slot_plies, d_status);
    SCB_CUDA(cudaGetLastError());
    return SC_OK;
}

int launch_path_replay(const void *d_root_rec, const int32_t *d_root_off, const int32_t *d_slot_plies,
                       const chess::Position *d_root_pos, const int32_t *d_root, const sc_move *d_path,
                       const int32_t *d_off, const int8_t *d_n_hist, int n, void *d_scratch, sc_position *d_pos,
                       int8_t *d_ep, int32_t *d_status, cudaStream_t st)
{
    if (n <= 0) return SC_OK;
    const dim3 grid((n + REPLAY_THREADS - 1) / REPLAY_THREADS);
    const ReplayPly *rec = static_cast<const ReplayPly *>(d_root_rec);
    ReplayPly *scratch = static_cast<ReplayPly *>(d_scratch);
    if (d_slot_plies)
        path_replay_kernel<<<grid, REPLAY_THREADS, 0, st>>>(rec, SlotRoots{d_slot_plies}, d_root_pos, d_root, d_path,
                                                            d_off, d_n_hist, n, scratch, d_pos, d_ep, d_status);
    else
        path_replay_kernel<<<grid, REPLAY_THREADS, 0, st>>>(rec, OffsetRoots{d_root_off}, d_root_pos, d_root, d_path,
                                                            d_off, d_n_hist, n, scratch, d_pos, d_ep, d_status);
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
