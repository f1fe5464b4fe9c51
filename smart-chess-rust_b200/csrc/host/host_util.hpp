// Host-side pieces shared by the batched driver (search.cpp) and the one-leaf-at-a-time mirror of the
// reference's `Game` interface (game.hpp): RNG, trace records + writer (src/trace.rs:5-42), and the
// packing of a game position with its history into the `sc_position` the device encoder reads.
#pragma once
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../../include/sc_b200.h"
#include "chess_rules.hpp"

namespace scb {
namespace host {
using namespace scb::chess;

// ---- deterministic per-tree RNG (splitmix64 / xoshiro256**) --------------------------------------
struct Rng {
    uint64_t s[4];
    static uint64_t splitmix(uint64_t &x)
    {
        uint64_t z = (x += 0x9E3779B97F4A7C15ULL);
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
        return z ^ (z >> 31);
    }
    void seed(uint64_t v)
    {
        for (int i = 0; i < 4; i++) s[i] = splitmix(v);
    }
    static uint64_t rotl(uint64_t x, int k) { return (x << k) | (x >> (64 - k)); }
    uint64_t next()
    {
        uint64_t r = rotl(s[1] * 5, 7) * 9, t = s[1] << 17;
        s[2] ^= s[0]; s[3] ^= s[1]; s[1] ^= s[2]; s[0] ^= s[3];
        s[2] ^= t;
        s[3] = rotl(s[3], 45);
        return r;
    }
    double uniform() { return (double)(next() >> 11) * (1.0 / 9007199254740992.0); }
    // single-precision stream for the Dirichlet noise (thousands of gamma draws per move and tree)
    float uniformf() { return ((float)(next() >> 40) + 0.5f) * (1.0f / 16777216.0f); }  // (0, 1)
    bool have_spare = false;
    float spare = 0.f;
    float normalf()
    {
        if (have_spare) {
            have_spare = false;
            return spare;
        }
        // Box-Muller, both outputs used
        const float u1 = uniformf(), u2 = uniformf();
        const float r = sqrtf(-2.0f * logf(u1));
        float sn, cs;
        sincosf(6.2831853f * u2, &sn, &cs);
        spare = r * sn;
        have_spare = true;
        return r * cs;
    }
    // Marsaglia-Tsang; alpha < 1 handled by the boost gamma(a) = gamma(a+1) * U^(1/a)
    float gammaf(float alpha)
    {
        float boost = 1.0f;
        if (alpha < 1.0f) {
            boost = expf(logf(uniformf()) / alpha);
            alpha += 1.0f;
        }
        const float d = alpha - 1.0f / 3.0f, c = 1.0f / sqrtf(9.0f * d);
        for (;;) {
            const float x = normalf();
            float v = 1.0f + c * x;
            if (v <= 0.f) continue;
            v = v * v * v;
            const float u = uniformf();
            const float x2 = x * x;
            if (u < 1.0f - 0.0331f * x2 * x2) return d * v * boost;
            if (logf(u) < 0.5f * x2 + d * (1.0f - v + logf(v))) return d * v * boost;
        }
    }
};

struct TraceStep {
    Move mv;
    float q;
    std::vector<Move> cmv;
    std::vector<int32_t> cn;
    std::vector<float> cq, cu;
};

struct TraceRec {
    std::vector<TraceStep> steps;
    int termination = T_NONE;
    int winner = -1;
    bool has_outcome = false;
};

inline const char *term_name(int t)
{
    switch (t) {
    case T_CHECKMATE: return "Checkmate";
    case T_STALEMATE: return "Stalemate";
    case T_INSUFFICIENT: return "InsufficientMaterial";
    case T_SEVENTYFIVE: return "SeventyfiveMoves";
    case T_FIVEFOLD: return "FivefoldRepetition";
    case T_FIFTY: return "FiftyMoves";
    case T_THREEFOLD: return "ThreefoldRepetition";
    default: return "VariantDraw";
    }
}

inline void append_float(std::string &s, float v)
{
    char b[48];
    if (v == (float)(long long)v && std::fabs(v) < 1e15f)
        snprintf(b, sizeof(b), "%.1f", (double)v);
    else
        snprintf(b, sizeof(b), "%.9g", (double)v);
    s += b;
}

// src/trace.rs:23-32: {"steps": [[move, q, [[move, n, q, uct], ...]], ...], "outcome": ...}
inline std::string trace_to_json(const TraceRec &t)
{
    std::string s = "{\"outcome\": ";
    if (t.has_outcome) {
        s += "{\"termination\": \"";
        s += term_name(t.termination);
        s += "\", \"winner\": ";
        s += t.winner == WHITE ? "\"White\"" : (t.winner == BLACK ? "\"Black\"" : "null");
        s += "}";
    } else
        s += "null";
    s += ", \"steps\": [";
    char u[8];
    for (size_t i = 0; i < t.steps.size(); i++) {
        const TraceStep &st = t.steps[i];
        if (i) s += ", ";
        uci(st.mv, u);
        s += "[\"";
        s += u;
        s += "\", ";
        append_float(s, st.q);
        s += ", [";
        for (size_t k = 0; k < st.cmv.size(); k++) {
            if (k) s += ", ";
            uci(st.cmv[k], u);
            s += "[\"";
            s += u;
            s += "\", ";
            s += std::to_string(st.cn[k]);
            s += ", ";
            append_float(s, st.cq[k]);
            s += ", ";
            append_float(s, st.cu[k]);
            s += "]";
        }
        s += "]]";
    }
    s += "]}";
    return s;
}

// ---- position-hash stand-in evaluator (test hook; same specification as the oracle's) ----------
inline uint64_t mix64(uint64_t x)
{
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    return x ^ (x >> 31);
}
inline uint64_t position_hash(const Position &p)
{
    uint64_t h = mix64(p.pt[PAWN]);
    h = mix64(h ^ p.pt[KNIGHT]);
    h = mix64(h ^ p.pt[BISHOP]);
    h = mix64(h ^ p.pt[ROOK]);
    h = mix64(h ^ p.pt[QUEEN]);
    h = mix64(h ^ p.pt[KING]);
    h = mix64(h ^ p.occ[WHITE]);
    h = mix64(h ^ (uint64_t)p.turn);
    h = mix64(h ^ p.clean_castling());
    h = mix64(h ^ (uint64_t)(p.ep + 1));
    return h;
}
inline float hash_eval(const Position &p, const Move *mv, int n, float *priors)
{
    const uint64_t h = position_hash(p);
    float sum = 0.f;
    for (int i = 0; i < n; i++) {
        uint64_t m = mix64(h ^ ((uint64_t)mv[i].from << 16) ^ ((uint64_t)mv[i].to << 8) ^ mv[i].promo);
        priors[i] = (float)((m >> 40) + 1) * (1.0f / 16777216.0f);
        sum += priors[i];
    }
    sum += 1e-5f;
    for (int i = 0; i < n; i++) priors[i] = priors[i] / sum;
    uint64_t v = mix64(h ^ 0xABCDEF);
    return ((float)(v >> 40) * (1.0f / 16777216.0f)) * 2.f - 1.f;
}

// The inputs of `_encode` (src/chess.rs:845-877) before rotation: up to `n_hist` most recent positions
// of the game (slot 0 = current) with their repetition flags, and the meta vector of the current one
// (`encode_meta`, src/chess.rs:652-662).
inline void pack_position(const Game &g, int n_hist, sc_position *out)
{
    if (n_hist > SC_LOOKBACK) n_hist = SC_LOOKBACK;
    if (n_hist > g.ply() + 1) n_hist = g.ply() + 1;
    memset(out->slot, 0, sizeof(out->slot));
    for (int k = 0; k < n_hist; k++) {
        const int ply = g.ply() - k;
        const Position &p = g.pos_at(ply);
        pack_slot(p.pt + 1, p.occ[WHITE], g.rep_at(ply), out->slot[k]);
    }
    pack_meta(g.cur, out->meta);
    out->n_hist = n_hist;
}

}  // namespace host
}  // namespace scb
