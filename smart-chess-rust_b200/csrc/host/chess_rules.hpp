// Native chess rules for the batched search driver (product code, host side).
//
// The reference reaches python-chess 1.11.1 through PyO3 for every board operation
// (src/chess.rs:665-788: legal_moves, push, outcome, move_stack, copy; src/chess.rs:356-412:
// turn, clocks, piece_map, is_repetition(2/3), castling rights).  This header provides the same
// operations natively, with the same observable semantics -- in particular the legal-move
// GENERATION ORDER of python-chess, which defines the child order of every tree node
// (src/backends/torch.rs:96,140-143) and therefore the tie-breaks of the search.
//
// Board representation: piece bitboards + colour occupancy, a1 = bit 0 ... h8 = bit 63;
// sliding attacks by directional rays and bit scans (classical ray attacks).
//
// The legal-move generator (attack tables, Position::gen_*, is_safe, gen_legal) also compiles for the device under
// nvcc: movegen.cu runs it one thread per leaf for sc_predict.  Generation order is defined here only, for both targets.
// The generator writes through a sink (anything with add(from, to, promo)): the host collects into a MoveList, a device
// thread writes straight into its leaf's output slot.
#pragma once
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <vector>

#include "../../../include/sc_b200.h"

#ifdef __CUDACC__
#define SCB_HD __host__ __device__ inline
#else
#define SCB_HD inline
#endif
// SCB_HD, always inlined in device code (the host build is left to the compiler)
#ifdef __CUDA_ARCH__
#define SCB_HD_DEVICE_INLINE __host__ __device__ __forceinline__
#else
#define SCB_HD_DEVICE_INLINE SCB_HD
#endif

namespace scb {
namespace chess {

typedef uint64_t u64;
enum { BLACK = 0, WHITE = 1 };
enum { NONE = 0, PAWN = 1, KNIGHT, BISHOP, ROOK, QUEEN, KING };
// src/chess.rs:87-105 `Termination`
enum { T_NONE = 0, T_CHECKMATE = 1, T_STALEMATE, T_INSUFFICIENT, T_SEVENTYFIVE, T_FIVEFOLD, T_FIFTY, T_THREEFOLD };

struct Move {
    uint8_t from, to, promo;
    bool operator==(const Move &o) const { return from == o.from && to == o.to && promo == o.promo; }
};

struct MoveList {
    Move m[256];
    int n = 0;
    SCB_HD void add(int f, int t, int p = 0)
    {
        m[n].from = (uint8_t)f;
        m[n].to = (uint8_t)t;
        m[n].promo = (uint8_t)p;
        n++;
    }
};

SCB_HD u64 bit(int s) { return 1ULL << s; }
#ifdef __CUDA_ARCH__
SCB_HD int lsb(u64 b) { return __ffsll((long long)b) - 1; }
SCB_HD int msb(u64 b) { return 63 - __clzll((long long)b); }
SCB_HD int popcnt(u64 b) { return __popcll(b); }
#else
inline int lsb(u64 b) { return __builtin_ctzll(b); }
inline int msb(u64 b) { return 63 - __builtin_clzll(b); }
inline int popcnt(u64 b) { return __builtin_popcountll(b); }
#endif
SCB_HD int rank_of(int s) { return s >> 3; }
SCB_HD int file_of(int s) { return s & 7; }
constexpr u64 RANK1 = 0xFFULL, RANK8 = 0xFFULL << 56, FILE_A = 0x0101010101010101ULL;
SCB_HD u64 rank_mask(int r) { return RANK1 << (8 * r); }

// direction order: N, S, E, W, NE, NW, SE, SW.  Plain data (70 KB): built once on the host, and copied as it is to the
// device (movegen.cu), where it is too large for constant memory.
struct Tables {
    u64 ray[8][64];
    u64 knight[64], king[64], pawn_att[2][64];
    u64 line[64][64];     // full line through a and b (edge to edge), 0 if not aligned
    u64 between[64][64];  // squares strictly between
    void build()
    {
        static const int dr[8] = {1, -1, 0, 0, 1, 1, -1, -1};
        static const int df[8] = {0, 0, 1, -1, 1, -1, 1, -1};
        for (int s = 0; s < 64; s++) {
            for (int d = 0; d < 8; d++) {
                u64 m = 0;
                int r = rank_of(s) + dr[d], f = file_of(s) + df[d];
                while (r >= 0 && r < 8 && f >= 0 && f < 8) {
                    m |= bit(r * 8 + f);
                    r += dr[d];
                    f += df[d];
                }
                ray[d][s] = m;
            }
            static const int kn[8][2] = {{2, 1}, {1, 2}, {-1, 2}, {-2, 1}, {-2, -1}, {-1, -2}, {1, -2}, {2, -1}};
            u64 a = 0, k = 0;
            for (int i = 0; i < 8; i++) {
                int r = rank_of(s) + kn[i][0], f = file_of(s) + kn[i][1];
                if (r >= 0 && r < 8 && f >= 0 && f < 8) a |= bit(r * 8 + f);
                r = rank_of(s) + dr[i];
                f = file_of(s) + df[i];
                if (r >= 0 && r < 8 && f >= 0 && f < 8) k |= bit(r * 8 + f);
            }
            knight[s] = a;
            king[s] = k;
            u64 w = 0, b = 0;
            for (int dfile = -1; dfile <= 1; dfile += 2) {
                int f = file_of(s) + dfile;
                if (f < 0 || f > 7) continue;
                if (rank_of(s) < 7) w |= bit(s + 8 + dfile);
                if (rank_of(s) > 0) b |= bit(s - 8 + dfile);
            }
            pawn_att[WHITE][s] = w;
            pawn_att[BLACK][s] = b;
        }
        for (int a = 0; a < 64; a++)
            for (int b = 0; b < 64; b++) {
                line[a][b] = 0;
                between[a][b] = 0;
                for (int d = 0; d < 8; d++)
                    if (ray[d][a] & bit(b)) {
                        int opp = d ^ 1;  // N<->S, E<->W, NE<->NW? no: pairs are (0,1),(2,3),(4,7),(5,6)
                        if (d >= 4) opp = 11 - d;
                        line[a][b] = ray[d][a] | ray[opp][a] | bit(a);
                        between[a][b] = ray[d][a] & ray[opp][b];
                    }
            }
    }
};

#ifdef __CUDACC__
// the device copy of the tables; defined by movegen.cu, the translation unit that generates moves on the device
__device__ const Tables &device_tables();
#endif

inline const Tables &host_tables()
{
    static const Tables t = [] {
        Tables x;
        x.build();
        return x;
    }();
    return t;
}

SCB_HD const Tables &T()
{
#ifdef __CUDA_ARCH__
    return device_tables();
#else
    return host_tables();
#endif
}

SCB_HD u64 ray_attack(int d, int s, u64 occ)
{
    const Tables &t = T();
    u64 r = t.ray[d][s];
    u64 blockers = r & occ;
    if (blockers) {
        // directions N, E, NE, NW increase the square index
        int first = (d == 0 || d == 2 || d == 4 || d == 5) ? lsb(blockers) : msb(blockers);
        r ^= t.ray[d][first];
    }
    return r;
}
SCB_HD u64 rook_attacks(int s, u64 occ) { return ray_attack(0, s, occ) | ray_attack(1, s, occ) | ray_attack(2, s, occ) | ray_attack(3, s, occ); }
SCB_HD u64 bishop_attacks(int s, u64 occ) { return ray_attack(4, s, occ) | ray_attack(5, s, occ) | ray_attack(6, s, occ) | ray_attack(7, s, occ); }
SCB_HD u64 rank_attacks(int s, u64 occ) { return ray_attack(2, s, occ) | ray_attack(3, s, occ); }

struct Position {
    u64 pt[7];  // [1..6] piece-type bitboards, both colours
    u64 occ[2];
    u64 all;
    u64 castling;  // rook squares that still carry the right
    int turn;
    int ep;  // en-passant square or -1
    int halfmove, fullmove;

    // the current board of a packed leaf: pieces and colour from slot[0] (white-oriented, unrotated), the side to move
    // from meta[0], castling rights from meta[2..5] (side to move K / Q, opponent K / Q) on the standard rook squares,
    // the en-passant square from `ep_square` (python-chess `ep_square`: -1, or the square a double push skipped)
    SCB_HD void set_packed(const sc_position &p, int ep_square)
    {
        all = 0;
        pt[NONE] = 0;
        for (int i = 0; i < 6; i++) {
            pt[PAWN + i] = p.slot[0][i];
            all |= p.slot[0][i];
        }
        occ[WHITE] = p.slot[0][6] & all;
        occ[BLACK] = all & ~occ[WHITE];
        turn = p.meta[0] ? WHITE : BLACK;
        const int us = turn, them = !us;
        const u64 k_rook[2] = {bit(63), bit(7)}, q_rook[2] = {bit(56), bit(0)};
        castling = (p.meta[2] ? k_rook[us] : 0) | (p.meta[3] ? q_rook[us] : 0) | (p.meta[4] ? k_rook[them] : 0) |
                   (p.meta[5] ? q_rook[them] : 0);
        ep = ep_square;
        halfmove = p.meta[6];
        fullmove = p.meta[1];
    }
    SCB_HD void set_start()
    {
        memset(this, 0, sizeof(*this));
        pt[PAWN] = rank_mask(1) | rank_mask(6);
        pt[KNIGHT] = bit(1) | bit(6) | bit(57) | bit(62);
        pt[BISHOP] = bit(2) | bit(5) | bit(58) | bit(61);
        pt[ROOK] = bit(0) | bit(7) | bit(56) | bit(63);
        pt[QUEEN] = bit(3) | bit(59);
        pt[KING] = bit(4) | bit(60);
        occ[WHITE] = rank_mask(0) | rank_mask(1);
        occ[BLACK] = rank_mask(6) | rank_mask(7);
        all = occ[WHITE] | occ[BLACK];
        castling = bit(0) | bit(7) | bit(56) | bit(63);
        turn = WHITE;
        ep = -1;
        halfmove = 0;
        fullmove = 1;
    }
    // Forsyth-Edwards notation (test hook: perft from the published test positions); false if malformed
    bool set_fen(const char *fen)
    {
        memset(this, 0, sizeof(*this));
        ep = -1;
        halfmove = 0;
        fullmove = 1;
        int r = 7, f = 0;
        const char *p = fen;
        for (; *p && *p != ' '; p++) {
            const char ch = *p;
            if (ch == '/') {
                r--;
                f = 0;
            } else if (ch >= '1' && ch <= '8')
                f += ch - '0';
            else {
                static const char *names = " pnbrqk";
                const char lo = (char)(ch | 0x20);
                const char *q = strchr(names + 1, lo);
                if (!q || r < 0 || f > 7) return false;
                const int color = ch == lo ? BLACK : WHITE;
                pt[q - names] |= bit(r * 8 + f);
                occ[color] |= bit(r * 8 + f);
                f++;
            }
        }
        all = occ[WHITE] | occ[BLACK];
        if (*p != ' ') return false;
        p++;
        turn = *p == 'w' ? WHITE : BLACK;
        p++;
        if (*p != ' ') return false;
        for (p++; *p && *p != ' '; p++) {
            if (*p == 'K') castling |= bit(7);
            if (*p == 'Q') castling |= bit(0);
            if (*p == 'k') castling |= bit(63);
            if (*p == 'q') castling |= bit(56);
        }
        if (*p != ' ') return false;
        p++;
        if (*p != '-') {
            if (p[0] < 'a' || p[0] > 'h' || p[1] < '1' || p[1] > '8') return false;
            ep = (p[1] - '1') * 8 + (p[0] - 'a');
            p++;
        }
        p++;
        if (*p == ' ') {
            int hm = 0, fm = 1;
            if (sscanf(p, " %d %d", &hm, &fm) >= 1) {
                halfmove = hm;
                fullmove = fm;
            }
        }
        return (pt[KING] & occ[WHITE]) && (pt[KING] & occ[BLACK]);
    }
    SCB_HD int piece_at(int s) const
    {
        u64 m = bit(s);
        if (!(all & m)) return NONE;
        for (int p = PAWN; p <= KING; p++)
            if (pt[p] & m) return p;
        return NONE;
    }
    SCB_HD int take(int s)
    {
        int p = piece_at(s);
        if (p) {
            u64 m = ~bit(s);
            pt[p] &= m;
            occ[0] &= m;
            occ[1] &= m;
            all &= m;
        }
        return p;
    }
    SCB_HD void put(int s, int p, int color)
    {
        take(s);
        u64 m = bit(s);
        pt[p] |= m;
        occ[color] |= m;
        all |= m;
    }
    SCB_HD int king_sq(int color) const
    {
        u64 k = pt[KING] & occ[color];
        return k ? msb(k) : -1;
    }
    SCB_HD u64 attackers(int color, int s, u64 occupied) const
    {
        const Tables &t = T();
        u64 rq = pt[ROOK] | pt[QUEEN], bq = pt[BISHOP] | pt[QUEEN];
        u64 a = (t.king[s] & pt[KING]) | (t.knight[s] & pt[KNIGHT]) | (rook_attacks(s, occupied) & rq) |
                (bishop_attacks(s, occupied) & bq) | (t.pawn_att[!color][s] & pt[PAWN]);
        return a & occ[color];
    }
    SCB_HD bool in_check() const
    {
        int k = king_sq(turn);
        return k >= 0 && attackers(!turn, k, all) != 0;
    }
    // python-chess clean_castling_rights (standard chess)
    SCB_HD u64 clean_castling() const
    {
        u64 c = castling & pt[ROOK];
        u64 w = c & occ[WHITE] & (bit(0) | bit(7));
        u64 b = c & occ[BLACK] & (bit(56) | bit(63));
        if (!(occ[WHITE] & pt[KING] & bit(4))) w = 0;
        if (!(occ[BLACK] & pt[KING] & bit(60))) b = 0;
        return w | b;
    }
    SCB_HD bool has_kingside(int color) const
    {
        u64 back = color == WHITE ? RANK1 : RANK8;
        if (!(pt[KING] & occ[color] & back)) return false;
        return (clean_castling() & back & bit(color == WHITE ? 7 : 63)) != 0;
    }
    SCB_HD bool has_queenside(int color) const
    {
        u64 back = color == WHITE ? RANK1 : RANK8;
        if (!(pt[KING] & occ[color] & back)) return false;
        return (clean_castling() & back & bit(color == WHITE ? 0 : 56)) != 0;
    }
    SCB_HD bool is_zeroing(const Move &m) const
    {
        u64 touched = bit(m.from) ^ bit(m.to);
        return (touched & pt[PAWN]) || (touched & occ[!turn]);
    }
    SCB_HD bool is_en_passant(const Move &m) const
    {
        int d = (int)m.to - (int)m.from;
        if (d < 0) d = -d;
        return ep == m.to && (pt[PAWN] & bit(m.from)) && (d == 7 || d == 9) && !(all & bit(m.to));
    }
    SCB_HD bool is_castling(const Move &m) const
    {
        if (!(pt[KING] & bit(m.from))) return false;
        int d = file_of(m.from) - file_of(m.to);
        return d > 1 || d < -1 || (pt[ROOK] & occ[turn] & bit(m.to));
    }

    // ---- python-chess Board.push ---------------------------------------------------------
    SCB_HD void push(const Move &m)
    {
        castling = clean_castling();
        const int old_ep = ep;
        ep = -1;
        halfmove++;
        if (turn == BLACK) fullmove++;
        if (is_zeroing(m)) halfmove = 0;
        const int us = turn;
        int p = take(m.from);
        int captured = piece_at(m.to);
        castling &= ~bit(m.from) & ~bit(m.to);
        if (p == KING) castling &= ~(us == WHITE ? RANK1 : RANK8);
        if (p == PAWN) {
            int diff = (int)m.to - (int)m.from;
            if (diff == 16 && rank_of(m.from) == 1) ep = m.from + 8;
            else if (diff == -16 && rank_of(m.from) == 6) ep = m.from - 8;
            else if (m.to == old_ep && (diff == 7 || diff == 9 || diff == -7 || diff == -9) && !captured)
                take(old_ep + (us == WHITE ? -8 : 8));
        }
        if (m.promo) p = m.promo;
        bool castled = false;
        if (p == KING) {
            int df = file_of(m.to) - file_of(m.from);
            if (df == 2 || df == -2) {
                int rook_from = (df < 0) ? (us == WHITE ? 0 : 56) : (us == WHITE ? 7 : 63);
                if (pt[ROOK] & occ[us] & bit(rook_from)) {
                    castled = true;
                    castling &= ~bit(rook_from);
                    take(rook_from);
                    put(m.to, KING, us);
                    put(df < 0 ? m.to + 1 : m.to - 1, ROOK, us);
                }
            }
        }
        if (!castled) put(m.to, p, us);
        turn = !us;
    }

    // ---- legal move generation in python-chess order ---------------------------------------
    SCB_HD u64 attacks_from(int s) const
    {
        const Tables &t = T();
        u64 m = bit(s);
        if (pt[PAWN] & m) return t.pawn_att[(occ[WHITE] & m) ? WHITE : BLACK][s];
        if (pt[KNIGHT] & m) return t.knight[s];
        if (pt[KING] & m) return t.king[s];
        u64 a = 0;
        if ((pt[BISHOP] | pt[QUEEN]) & m) a |= bishop_attacks(s, all);
        if ((pt[ROOK] | pt[QUEEN]) & m) a |= rook_attacks(s, all);
        return a;
    }
    template <class Sink> SCB_HD static void add_pawn(Sink &l, int from, int to)
    {
        int r = rank_of(to);
        if (r == 0 || r == 7) {
            l.add(from, to, QUEEN);
            l.add(from, to, ROOK);
            l.add(from, to, BISHOP);
            l.add(from, to, KNIGHT);
        } else
            l.add(from, to, 0);
    }
    template <class Sink> SCB_HD void gen_ep(u64 from_mask, u64 to_mask, Sink &l) const
    {
        if (ep < 0 || !(bit(ep) & to_mask) || (bit(ep) & all)) return;
        u64 c = pt[PAWN] & occ[turn] & from_mask & T().pawn_att[!turn][ep] & rank_mask(turn == WHITE ? 4 : 3);
        while (c) {
            int s = msb(c);
            c ^= bit(s);
            l.add(s, ep, 0);
        }
    }
    SCB_HD bool any_attacked(u64 squares, u64 occupied) const
    {
        while (squares) {
            int s = msb(squares);
            squares ^= bit(s);
            if (attackers(!turn, s, occupied)) return true;
        }
        return false;
    }
    template <class Sink> SCB_HD void gen_castling(u64 from_mask, u64 to_mask, Sink &l) const
    {
        const Tables &t = T();
        u64 back = turn == WHITE ? RANK1 : RANK8;
        u64 king = occ[turn] & pt[KING] & back & from_mask;
        king &= -king;
        if (!king) return;
        int ks = msb(king);
        u64 cands = clean_castling() & back & to_mask;
        while (cands) {
            int rs = msb(cands);
            cands ^= bit(rs);
            u64 rook = bit(rs);
            bool a_side = rook < king;
            int kto = (turn == WHITE ? 0 : 56) + (a_side ? 2 : 6);
            int rto = (turn == WHITE ? 0 : 56) + (a_side ? 3 : 5);
            u64 kpath = t.between[ks][kto], rpath = t.between[rs][rto];
            if ((all ^ king ^ rook) & (kpath | rpath | bit(kto) | bit(rto))) continue;
            if (any_attacked(kpath | king, all ^ king)) continue;
            if (any_attacked(bit(kto), all ^ king ^ rook ^ bit(rto))) continue;
            l.add(ks, kto, 0);
        }
    }
    template <class Sink> SCB_HD void gen_pseudo(u64 from_mask, u64 to_mask, Sink &l) const
    {
        const Tables &t = T();
        u64 ours = occ[turn];
        u64 pieces = ours & ~pt[PAWN] & from_mask;
        while (pieces) {
            int s = msb(pieces);
            pieces ^= bit(s);
            u64 mv = attacks_from(s) & ~ours & to_mask;
            while (mv) {
                int d = msb(mv);
                mv ^= bit(d);
                l.add(s, d, 0);
            }
        }
        if (from_mask & pt[KING]) gen_castling(from_mask, to_mask, l);
        u64 pawns = pt[PAWN] & ours & from_mask;
        if (!pawns) return;
        u64 caps = pawns;
        while (caps) {
            int s = msb(caps);
            caps ^= bit(s);
            u64 tg = t.pawn_att[turn][s] & occ[!turn] & to_mask;
            while (tg) {
                int d = msb(tg);
                tg ^= bit(d);
                add_pawn(l, s, d);
            }
        }
        u64 single, dbl;
        if (turn == WHITE) {
            single = (pawns << 8) & ~all;
            dbl = (single << 8) & ~all & (rank_mask(2) | rank_mask(3));
        } else {
            single = (pawns >> 8) & ~all;
            dbl = (single >> 8) & ~all & (rank_mask(5) | rank_mask(4));
        }
        single &= to_mask;
        dbl &= to_mask;
        const int back1 = turn == WHITE ? -8 : 8;
        while (single) {
            int d = msb(single);
            single ^= bit(d);
            add_pawn(l, d + back1, d);
        }
        while (dbl) {
            int d = msb(dbl);
            dbl ^= bit(d);
            l.add(d + 2 * back1, d, 0);
        }
        if (ep >= 0) gen_ep(from_mask, to_mask, l);
    }
    SCB_HD u64 slider_blockers(int king) const
    {
        const Tables &t = T();
        u64 rq = pt[ROOK] | pt[QUEEN], bq = pt[BISHOP] | pt[QUEEN];
        u64 snipers = ((rook_attacks(king, 0) & rq) | (bishop_attacks(king, 0) & bq)) & occ[!turn];
        u64 blockers = 0;
        while (snipers) {
            int s = msb(snipers);
            snipers ^= bit(s);
            u64 b = t.between[king][s] & all;
            if (b && !(b & (b - 1))) blockers |= b;
        }
        return blockers & occ[turn];
    }
    SCB_HD u64 pin_mask(int color, int s) const
    {
        const Tables &t = T();
        int king = king_sq(color);
        if (king < 0) return ~0ULL;
        u64 sm = bit(s);
        u64 rq = pt[ROOK] | pt[QUEEN], bq = pt[BISHOP] | pt[QUEEN];
        u64 rays[3] = {ray_attack(0, king, 0) | ray_attack(1, king, 0), rank_attacks(king, 0), bishop_attacks(king, 0)};
        u64 sl[3] = {rq, rq, bq};
        for (int i = 0; i < 3; i++)
            if (rays[i] & sm) {
                u64 snipers = rays[i] & sl[i] & occ[!color];
                while (snipers) {
                    int sn = msb(snipers);
                    snipers ^= bit(sn);
                    if ((t.between[sn][king] & (all | sm)) == sm) return t.line[king][sn];
                }
                break;
            }
        return ~0ULL;
    }
    SCB_HD bool ep_skewered(int king, int capturer) const
    {
        int last_double = ep + (turn == WHITE ? -8 : 8);
        u64 o = (all & ~bit(last_double) & ~bit(capturer)) | bit(ep);
        if (rank_attacks(king, o) & occ[!turn] & (pt[ROOK] | pt[QUEEN])) return true;
        if (bishop_attacks(king, o) & occ[!turn] & (pt[BISHOP] | pt[QUEEN])) return true;
        return false;
    }
    SCB_HD bool is_safe(int king, u64 blockers, const Move &m) const
    {
        if (m.from == king) {
            if (is_castling(m)) return true;
            return !attackers(!turn, m.to, all);
        }
        if (is_en_passant(m)) return (pin_mask(turn, m.from) & bit(m.to)) && !ep_skewered(king, m.from);
        return !(blockers & bit(m.from)) || (T().line[m.from][m.to] & bit(king));
    }
    template <class Sink> SCB_HD void gen_evasions(int king, u64 checkers, Sink &l) const
    {
        const Tables &t = T();
        u64 sliders = checkers & (pt[BISHOP] | pt[ROOK] | pt[QUEEN]);
        u64 attacked = 0;
        while (sliders) {
            int c = msb(sliders);
            sliders ^= bit(c);
            attacked |= t.line[king][c] & ~bit(c);
        }
        u64 mv = t.king[king] & ~occ[turn] & ~attacked;
        while (mv) {
            int d = msb(mv);
            mv ^= bit(d);
            l.add(king, d, 0);
        }
        int checker = msb(checkers);
        if (bit(checker) == checkers) {
            u64 target = t.between[king][checker] | checkers;
            gen_pseudo(~pt[KING], target, l);
            if (ep >= 0 && !(bit(ep) & target)) {
                int last_double = ep + (turn == WHITE ? -8 : 8);
                if (last_double == checker) gen_ep(~0ULL, ~0ULL, l);
            }
        }
    }
    // passes the pseudo-legal candidates that is_safe accepts on to `out`, in generation order (without a king to keep
    // safe, king < 0, every candidate)
    template <class Sink> struct SafeFilter {
        const Position &p;
        int king;
        u64 blockers;
        Sink &out;
        int seen;  // pseudo-legal candidates generated
        SCB_HD void add(int f, int t, int pr)
        {
            seen++;
            const Move m{(uint8_t)f, (uint8_t)t, (uint8_t)pr};
            if (king < 0 || p.is_safe(king, blockers, m)) out.add(f, t, pr);
        }
    };
    // the legal moves in python-chess order into `out`; returns the number of pseudo-legal candidates they were
    // filtered from (never fewer than the legal moves)
    // always inlined on the device: has_legal_ep's instance is reached from both replay kernels of movegen.cu (through
    // tkey), and left a call it costs the leaf replay kernel 64 B of spill stores
    template <class Sink> SCB_HD_DEVICE_INLINE int gen_legal(Sink &out) const
    {
        const int king = king_sq(turn);
        SafeFilter<Sink> f{*this, king, 0, out, 0};
        u64 checkers = 0;
        if (king >= 0) {
            f.blockers = slider_blockers(king);
            checkers = attackers(!turn, king, all);
        }
        if (checkers)
            gen_evasions(king, checkers, f);
        else
            gen_pseudo(~0ULL, ~0ULL, f);
        return f.seen;
    }
    void legal_moves(MoveList &out) const
    {
        out.n = 0;
        gen_legal(out);
    }
    // sinks of has_legal_ep: whether any move is generated, whether an en-passant capture is
    struct AnySink {
        bool any;
        SCB_HD void add(int, int, int) { any = true; }
    };
    struct EpSink {
        const Position &p;
        bool any;
        SCB_HD void add(int f, int t, int pr) { any = any || p.is_en_passant(Move{(uint8_t)f, (uint8_t)t, (uint8_t)pr}); }
    };
    SCB_HD bool has_legal_ep() const
    {
        if (ep < 0) return false;
        AnySink c{false};
        gen_ep(~0ULL, ~0ULL, c);
        if (!c.any) return false;
        EpSink l{*this, false};
        gen_legal(l);
        return l.any;
    }
    SCB_HD bool reduces_castling(const Move &m) const
    {
        u64 cr = clean_castling();
        u64 touched = bit(m.from) ^ bit(m.to);
        return (touched & cr) || ((cr & RANK1) && (touched & pt[KING] & occ[WHITE])) ||
               ((cr & RANK8) && (touched & pt[KING] & occ[BLACK]));
    }
    SCB_HD bool is_irreversible(const Move &m) const { return is_zeroing(m) || reduces_castling(m) || has_legal_ep(); }
    bool insufficient(int color) const
    {
        u64 own = occ[color];
        if (own & (pt[PAWN] | pt[ROOK] | pt[QUEEN])) return false;
        if (own & pt[KNIGHT]) return popcnt(own) <= 2 && !(occ[!color] & ~pt[KING] & ~pt[QUEEN]);
        if (own & pt[BISHOP]) {
            const u64 dark = 0xAA55AA55AA55AA55ULL, light = 0x55AA55AA55AA55AAULL;
            bool same = !(pt[BISHOP] & dark) || !(pt[BISHOP] & light);
            return same && !pt[PAWN] && !pt[KNIGHT];
        }
        return true;
    }
};

// transposition key of python-chess (_transposition_key)
struct TKey {
    u64 pt[6], w, b, cr;
    int turn, ep;
    SCB_HD bool operator==(const TKey &o) const
    {
        for (int i = 0; i < 6; i++)
            if (pt[i] != o.pt[i]) return false;
        return w == o.w && b == o.b && cr == o.cr && turn == o.turn && ep == o.ep;
    }
};
SCB_HD TKey tkey(const Position &p)
{
    TKey k;
    for (int i = 0; i < 6; i++) k.pt[i] = p.pt[i + 1];
    k.w = p.occ[WHITE];
    k.b = p.occ[BLACK];
    k.cr = p.clean_castling();
    k.turn = p.turn;
    k.ep = p.has_legal_ep() ? p.ep : -1;
    return k;
}

// The packed form of a leaf (`_encode`'s inputs, src/chess.rs:845-877): one history slot, the piece-type boards
// pieces[0..5] (pawn .. king) and White's occupancy of a position with its repetition flags `rep` (bit 0
// is_repetition(2), bit 1 is_repetition(3)), and the meta vector of the current position (`encode_meta`,
// src/chess.rs:652-662).  host::pack_position and the device replay of sc_predict_stack both write them.
SCB_HD void pack_slot(const u64 *pieces, u64 white, u64 rep, uint64_t *s)
{
    for (int i = 0; i < 6; i++) s[i] = pieces[i];
    s[6] = white;
    s[7] = rep;
}
SCB_HD void pack_meta(const Position &c, int32_t *meta)
{
    meta[0] = c.turn;
    meta[1] = c.fullmove;
    meta[2] = c.has_kingside(c.turn);
    meta[3] = c.has_queenside(c.turn);
    meta[4] = c.has_kingside(!c.turn);
    meta[5] = c.has_queenside(!c.turn);
    meta[6] = c.halfmove;
}

// python-chess Board.is_repetition(count) of the position after `ply` moves, whose halfmove clock is `halfmove`, over a
// history with h.occupancy(k) / h.key(k) = the occupied squares / tkey of the position after k moves (k <= ply) and
// h.irreversible(k) = whether move k is irreversible (k < ply).  The host Game and the device replay of
// sc_predict_stack (movegen.cu) both call it, so the repetition flags of a packed leaf are defined in one place.
#ifdef __CUDACC__
#pragma nv_exec_check_disable  // the host Game's accessor is host code; the device instantiation has a device one
#endif
template <class History> SCB_HD bool is_repetition(const History &h, int ply, int halfmove, int count)
{
    // python-chess pre-filters on equal occupancy over the whole stack; the exact walk below stops at
    // the first irreversible move, and every zeroing move is irreversible, so only the last
    // `halfmove` plies can hold a real repetition -- scanning just those gives the same answer
    int maybe = 1;
    const u64 all = h.occupancy(ply);
    const int lo = ply - halfmove > 0 ? ply - halfmove : 0;
    for (int k = ply - 1; k >= lo; k--)
        if (h.occupancy(k) == all && ++maybe >= count) break;
    if (maybe < count) return false;
    const TKey key = h.key(ply);
    int len = ply;
    for (;;) {
        if (count <= 1) return true;
        if (len < count - 1) break;
        len--;
        if (h.irreversible(len)) break;
        if (h.key(len) == key) count--;
    }
    return false;
}

// A game = python-chess Board with its move stack (`BoardState`, src/chess.rs:107-109).  Every
// stack entry caches the two repetition flags of `Board::extract` for that position, so packing
// the 8-slot history of a leaf never replays the game (the reference memoises this with a
// 50 000-entry cache, src/chess.rs:553-591).
struct Game {
    struct Entry {
        Position pos;  // position BEFORE moves[i]
        uint8_t rep;   // bit 0 is_repetition(2), bit 1 is_repetition(3) of `pos`
    };
    Position cur;
    uint8_t cur_rep = 0;
    std::vector<Entry> stack;
    std::vector<Move> moves;

    Game() { cur.set_start(); }
    int ply() const { return (int)moves.size(); }
    const Position &pos_at(int k) const { return k == ply() ? cur : stack[k].pos; }
    uint8_t rep_at(int k) const { return k == ply() ? cur_rep : stack[k].rep; }

    // the history accessor of chess::is_repetition
    u64 occupancy(int k) const { return pos_at(k).all; }
    TKey key(int k) const { return tkey(pos_at(k)); }
    bool irreversible(int k) const { return stack[k].pos.is_irreversible(moves[k]); }
    bool is_repetition(int count) const { return chess::is_repetition(*this, ply(), cur.halfmove, count); }
    void push(const Move &m)
    {
        stack.push_back(Entry{cur, cur_rep});
        moves.push_back(m);
        cur.push(m);
        // three occurrences imply two
        cur_rep = is_repetition(2) ? (uint8_t)(1 | (is_repetition(3) ? 2 : 0)) : (uint8_t)0;
    }
    void pop()
    {
        cur = stack.back().pos;
        cur_rep = stack.back().rep;
        stack.pop_back();
        moves.pop_back();
    }
    // python-chess outcome(claim_draw); winner: WHITE/BLACK or -1
    int outcome(bool claim_draw, int *winner)
    {
        MoveList l;
        cur.legal_moves(l);
        *winner = -1;
        if (l.n == 0 && cur.in_check()) {
            *winner = !cur.turn;
            return T_CHECKMATE;
        }
        if (cur.insufficient(WHITE) && cur.insufficient(BLACK)) return T_INSUFFICIENT;
        if (l.n == 0) return T_STALEMATE;
        if (cur.halfmove >= 150) return T_SEVENTYFIVE;
        if (is_repetition(5)) return T_FIVEFOLD;
        if (!claim_draw) return T_NONE;
        if (cur.halfmove >= 100) return T_FIFTY;
        if (cur.halfmove >= 99)
            for (int i = 0; i < l.n; i++)
                if (!cur.is_zeroing(l.m[i])) {
                    Position nx = cur;
                    nx.push(l.m[i]);
                    MoveList l2;
                    nx.legal_moves(l2);
                    if (l2.n > 0) return T_FIFTY;
                }
        std::vector<TKey> keys;
        keys.push_back(tkey(cur));
        for (int len = ply(); len > 0;) {
            len--;
            if (stack[len].pos.is_irreversible(moves[len])) break;
            keys.push_back(tkey(stack[len].pos));
        }
        int cnt = 0;
        for (auto &k : keys) cnt += k == keys[0];
        if (cnt >= 3) return T_THREEFOLD;
        for (int i = 0; i < l.n; i++) {
            Position nx = cur;
            nx.push(l.m[i]);
            TKey nk = tkey(nx);
            int c2 = 0;
            for (auto &k : keys) c2 += k == nk;
            if (c2 >= 2) return T_THREEFOLD;
        }
        return T_NONE;
    }
};

inline void uci(const Move &m, char *out)
{
    static const char *pc = " pnbrqk";
    out[0] = (char)('a' + file_of(m.from));
    out[1] = (char)('1' + rank_of(m.from));
    out[2] = (char)('a' + file_of(m.to));
    out[3] = (char)('1' + rank_of(m.to));
    out[4] = m.promo ? pc[m.promo] : 0;
    out[5] = 0;
}

}  // namespace chess
}  // namespace scb
