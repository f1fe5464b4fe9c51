// `sc_game_selfplay`: one self-play game through the C++ mirror of the reference's own interface
// (host/game.hpp): `mcts::mcts` -> `select` -> `Game::predict` one leaf at a time, `mcts::step`, and the
// move loop of src/main.rs:153-238.  This is the path a `selfplay` binary built against the new backend
// takes; the batched driver (search.cpp) is the throughput path and must produce the same games.
// `sc_game_selfplay_many` plays many such games on host threads through one batching evaluator (host/evaluator.cpp).
#include <cstring>
#include <functional>
#include <string>
#include <thread>

#include "../common.cuh"
#include "evaluator.hpp"
#include "game.hpp"

using namespace smartchess;

namespace {

// evaluator stand-in with the specification of the oracle's hash evaluator (CPU tests)
class ChessHash : public Game<BoardState> {
public:
    std::tuple<std::vector<Step>, std::vector<float>, float> predict(const ArcRefNode<Step> &node, const BoardState &state,
                                                                      bool) const override
    {
        const std::vector<Move> legal = state.legal_moves();
        if (legal.empty()) {
            float v = 0.f;
            if (state.is_check()) v = state.turn() == Color::White ? -1.f : 1.f;
            return {{}, {}, v};
        }
        std::vector<float> priors(legal.size());
        const float value = scb::host::hash_eval(state.game().cur, legal.data(), (int)legal.size(), priors.data());
        std::vector<Step> steps;
        for (const Move &m : legal) steps.push_back(Step{m, !node->step.color});
        return {std::move(steps), std::move(priors), value};
    }
    bool reverse_q(const ArcRefNode<Step> &node) const override { return node->step.color == Color::Black; }
};

std::optional<std::vector<float>> dirichlet_noise(size_t size, void *ctx)
{
    if (size < 2) return std::nullopt;
    scb::host::Rng *rng = static_cast<scb::host::Rng *>(ctx);
    std::vector<float> g(size);
    float tot = 0.f;
    for (auto &x : g) tot += (x = rng->gammaf(0.3f));
    for (auto &x : g) x /= tot;
    return g;
}

double uniform01(void *ctx) { return static_cast<scb::host::Rng *>(ctx)->uniform(); }

// one game of src/main.rs:153-238 through `chess` with the RNG seeded from `seed`: the trace as JSON.  before_search
// (may be null) sees each search root before its search
std::string play_game(const Game<BoardState> &chess, const sc_selfplay_config &cfg, uint64_t seed,
                      const std::function<void(const BoardState &)> &before_search)
{
    scb::host::Rng rng;
    rng.seed(seed * 0x9E3779B97F4A7C15ULL + 1);
    scb::host::TraceRec trace;
    BoardState state;
    Node<Step> root_node;
    root_node.step = Step{std::nullopt, Color::White};
    auto [cursor, root] = Cursor<Step>::create(std::move(root_node));
    std::optional<Outcome> outcome;
    for (int i = 0; i < cfg.num_steps; i++) {
        const float temperature = i < cfg.temperature_switch ? 1.0f : cfg.temperature;
        // src/main.rs:175-180
        const int rollout = cfg.rollout_factor > 0.f
                                ? std::min(300, (int)((float)state.legal_moves().size() * cfg.rollout_factor))
                                : (cfg.rollout_num > 0 ? cfg.rollout_num : 300);
        if (before_search) before_search(state);
        mcts::mcts<Game<BoardState>, BoardState>(chess, cursor.arc(), state, rollout, cfg.cpuct, cfg.epsilon,
                                                 cfg.with_noise != 0, dirichlet_noise, &rng);
        scb::host::TraceStep st;
        st.q = cursor.current().q_value;
        for (const auto &n : cursor.current().children) {
            st.cmv.push_back(*n->step.mv);
            st.cn.push_back(n->num_act);
            st.cq.push_back(n->q_value);
            st.cu.push_back(n->uct);
        }
        const auto played = mcts::step<BoardState>(cursor, state, temperature, uniform01, &rng);
        if (!played) {
            outcome = state.outcome();
            break;
        }
        st.mv = *played->mv;
        trace.steps.push_back(std::move(st));
        if (i > 100) {
            outcome = state.outcome();
            if (outcome) break;
        }
    }
    if (outcome) {
        trace.has_outcome = true;
        trace.termination = outcome->termination;
        trace.winner = outcome->winner ? (int)*outcome->winner : -1;
    }
    return scb::host::trace_to_json(trace);
}

// copies s (cut to cap - 1 bytes) with its NUL to buf; the bytes s needs
int64_t copy_trace(const std::string &s, char *buf, int64_t cap)
{
    if (buf && cap > 0) {
        const int64_t n = std::min<int64_t>(cap - 1, (int64_t)s.size());
        memcpy(buf, s.data(), (size_t)n);
        buf[n] = 0;
    }
    return (int64_t)s.size() + 1;
}

bool bad_config(const sc_selfplay_config *cfg, const sc_engine *e)
{
    return !cfg || cfg->rollout_num < 0 || cfg->rollout_factor < 0.f || (cfg->rollout_num > 0 && cfg->rollout_factor > 0.f) ||
           cfg->num_steps <= 0 || (cfg->evaluator == 0 && !e) || (cfg->evaluator != 0 && cfg->evaluator != 1);
}

}  // namespace

extern "C" int64_t sc_game_selfplay(sc_engine *e, const sc_selfplay_config *cfg, char *buf, int64_t cap)
{
    if (bad_config(cfg, e)) {
        scb::set_error("sc_game_selfplay: bad argument");
        return -1;
    }
    try {
        std::unique_ptr<Game<BoardState>> chess;
        if (cfg->evaluator == 0)
            chess.reset(new ChessB200(e));
        else
            chess.reset(new ChessHash());
        return copy_trace(play_game(*chess, *cfg, cfg->seed, nullptr), buf, cap);
    } catch (const std::exception &ex) {
        scb::set_error(std::string("sc_game_selfplay: ") + ex.what());
        return -1;
    }
}

extern "C" int sc_game_selfplay_many(sc_engine *e, const sc_selfplay_config *cfg, int n_games, const uint64_t *seeds,
                                     char *buf, int64_t cap, int64_t *sizes, sc_evaluator_counts *counts_out)
{
    if (bad_config(cfg, e) || n_games < 1 || !seeds || !sizes || (buf && cap <= 0)) {
        scb::set_error("sc_game_selfplay_many: bad argument");
        return SC_E_INVAL;
    }
    sc_evaluator *ev = nullptr;
    if (cfg->evaluator == 0)
        SCB_CHECK(sc_evaluator_create(e, n_games, &ev));
    else
        SCB_CHECK(scb::evaluator_create(scb::hash_backend_create(n_games), n_games, n_games, &ev));
    std::vector<std::string> err((size_t)n_games);
    std::vector<std::thread> games;
    games.reserve((size_t)n_games);
    for (int g = 0; g < n_games; g++)
        games.emplace_back([&, g] {
            try {
                ChessB200Slot chess(ev, g);
                const std::string s = play_game(chess, *cfg, seeds[g], [&](const BoardState &st) { chess.set_search_root(st); });
                sizes[g] = copy_trace(s, buf ? buf + (int64_t)g * cap : nullptr, cap);
            } catch (const std::exception &ex) {
                sizes[g] = -1;
                err[g] = std::string("sc_game_selfplay_many: game ") + std::to_string(g) + ": " + ex.what();
            }
        });
    for (std::thread &t : games) t.join();
    if (counts_out) sc_evaluator_stats(ev, counts_out);
    sc_evaluator_destroy(ev);
    for (int g = 0; g < n_games; g++)
        if (!err[g].empty()) {
            scb::set_error(err[g]);
            return SC_E_INVAL;
        }
    return SC_OK;
}
