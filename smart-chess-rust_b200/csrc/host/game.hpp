// C++ mirror of the reference's evaluator plug-in interface and of the one-leaf-at-a-time search that
// calls it.  Rust is not available in the build image, so this is the host side a Rust maintainer
// would otherwise write in `src/backends/b200.rs` (INTEGRATION.md): same names, same argument
// meaning, same error behaviour (the reference panics; here: std::runtime_error).
//
//   trait Game<S: State> { predict, reverse_q }            src/game.rs:3-15
//   trait State { type Step; dup; advance }                src/game.rs:17-21
//   Node<T>, ArcRefNode<T>, Cursor<T>                      src/mcts.rs:13-24, 59, 330-396
//   uct, find_max, backward, select, mcts, step            src/mcts.rs:61-98, 132-328
//   Step(Option<Move>, Color), BoardState                  src/chess.rs:65-66, 665-788
//   ChessB200::predict  ==  chess_tch_predict              src/backends/torch.rs:89-146
//
// `select` calls `predict` at EVERY level of every descent, as the reference does; the batched driver
// (search.cpp) stores the priors at expansion instead.  Both produce the same trees
// (tests/test_gpu_selfplay.py::test_game_interface_mirror_*).
#pragma once
#include <cmath>
#include <deque>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <tuple>
#include <vector>

#include "../../../include/sc_b200.h"
#include "chess_rules.hpp"
#include "host_util.hpp"

namespace smartchess {

using scb::chess::Move;
enum class Color : int { Black = scb::chess::BLACK, White = scb::chess::WHITE };
inline Color operator!(Color c) { return c == Color::White ? Color::Black : Color::White; }

// ---- src/mcts.rs:13-24 -----------------------------------------------------------------------------
template <class T> struct Node;
template <class T> using ArcRefNode = std::shared_ptr<Node<T>>;
template <class T> using WeakRefNode = std::weak_ptr<Node<T>>;

template <class T> struct Node {
    T step;
    uint32_t depth = 0;
    float q_value = 0.f;
    int32_t num_act = 0;
    float uct = 0.f;
    std::optional<WeakRefNode<T>> parent;
    std::vector<ArcRefNode<T>> children;

    void reset()  // src/mcts.rs:229-235: the parent link and the depth stay
    {
        q_value = 0.f;
        num_act = 0;
        children.clear();
    }
};

// ---- src/mcts.rs:59, 330-396 -----------------------------------------------------------------------
template <class T> class Cursor {
    ArcRefNode<T> p_;

public:
    explicit Cursor(ArcRefNode<T> arc) : p_(std::move(arc)) {}
    static std::pair<Cursor, ArcRefNode<T>> create(Node<T> data)  // `Cursor::new`: the caller keeps the root alive
    {
        auto arc = std::make_shared<Node<T>>(std::move(data));
        return {Cursor(arc), arc};
    }
    static Cursor from_arc(ArcRefNode<T> arc) { return Cursor(std::move(arc)); }
    const Node<T> &current() const { return *p_; }
    Node<T> &current_mut() { return *p_; }
    const ArcRefNode<T> &arc() const { return p_; }
    void navigate_down(size_t index)
    {
        if (index >= p_->children.size()) throw std::runtime_error("navigating to an nonexistent child.");
        p_ = p_->children[index];
    }
    void navigate_up()
    {
        if (!p_->parent) throw std::runtime_error("navigating to the parent, but already at the root");
        auto up = p_->parent->lock();
        if (!up) throw std::runtime_error("navigating to the parent, but failed to turn the weak ref into an arc");
        p_ = up;
    }
};

// ---- src/game.rs:3-21 ------------------------------------------------------------------------------
template <class S> struct Game {
    using Step = typename S::Step;
    virtual ~Game() = default;
    // (legal steps in generation order, their priors, value from White's point of view)
    virtual std::tuple<std::vector<Step>, std::vector<float>, float> predict(const ArcRefNode<Step> &node, const S &state,
                                                                              bool argmax) const = 0;
    virtual bool reverse_q(const ArcRefNode<Step> &node) const = 0;
};

// ---- src/chess.rs:65-66, 665-788 -------------------------------------------------------------------
struct Step {
    std::optional<Move> mv;  // None only at the root of a game
    Color color;             // the side to move AFTER the move
};

struct Outcome {
    int termination;               // scb::chess::T_*
    std::optional<Color> winner;
};

class BoardState {
    scb::chess::Game g_;

public:
    using Step = smartchess::Step;
    BoardState() = default;
    BoardState dup() const { return *this; }
    void advance(const Step &s)  // `next` (src/chess.rs:775-783)
    {
        if (!s.mv) throw std::runtime_error("advance: step without a move");
        g_.push(*s.mv);
    }
    std::vector<Move> legal_moves() const
    {
        scb::chess::MoveList l;
        g_.cur.legal_moves(l);
        return std::vector<Move>(l.m, l.m + l.n);
    }
    std::optional<Outcome> outcome()  // python-chess outcome(claim_draw=True), src/chess.rs:719-729
    {
        int w;
        const int t = g_.outcome(true, &w);
        if (t == scb::chess::T_NONE) return std::nullopt;
        Outcome o{t, std::nullopt};
        if (w >= 0) o.winner = w == scb::chess::WHITE ? Color::White : Color::Black;
        return o;
    }
    const std::vector<Move> &move_stack() const { return g_.moves; }
    Color turn() const { return g_.cur.turn == scb::chess::WHITE ? Color::White : Color::Black; }
    bool is_check() const { return g_.cur.in_check(); }
    const scb::chess::Game &game() const { return g_; }
};

// ---- the new backend: src/backends/torch.rs:14-52, 89-180 with the device doing encode + net + gather -
class ChessB200 : public Game<BoardState> {
    sc_engine *engine_;

public:
    explicit ChessB200(sc_engine *engine) : engine_(engine)
    {
        if (!engine) throw std::runtime_error("ChessB200: null engine");
    }

    std::tuple<std::vector<Step>, std::vector<float>, float> predict(const ArcRefNode<Step> &node, const BoardState &state,
                                                                      bool argmax) const override
    {
        if (argmax) throw std::runtime_error("predict: argmax is not used by mcts and not implemented");
        const std::vector<Move> legal = state.legal_moves();
        if (legal.empty()) {  // terminal: no network call (torch.rs:98-106)
            float v = 0.f;
            if (state.is_check()) v = state.turn() == Color::White ? -1.f : 1.f;
            return {{}, {}, v};
        }
        const Color turn = node->step.color;
        if (turn != state.turn()) throw std::runtime_error("predict: node and state disagree on the side to move");  // torch.rs:111
        // history: this node and up to 7 ancestors (`_encode`, chess.rs:845-867)
        int n_hist = 0;
        for (ArcRefNode<Step> n = node; n && n_hist < SC_LOOKBACK;) {
            n_hist++;
            if (!n->parent) break;
            n = n->parent->lock();
        }
        if (n_hist > (int)state.move_stack().size() + 1) throw std::runtime_error("predict: history longer than the move stack");  // chess.rs:863
        sc_position pos;
        scb::host::pack_position(state.game(), n_hist, &pos);
        std::vector<sc_move> moves(legal.size());
        for (size_t i = 0; i < legal.size(); i++) moves[i] = sc_move{legal[i].from, legal[i].to, legal[i].promo, 0};
        const int32_t off[2] = {0, (int32_t)legal.size()};
        std::vector<float> priors(legal.size());
        float value = 0.f;
        if (sc_eval(engine_, 1, &pos, moves.data(), off, priors.data(), &value, nullptr) != SC_OK)
            throw std::runtime_error(std::string("sc_eval: ") + sc_last_error());
        std::vector<Step> steps;
        steps.reserve(legal.size());
        for (const Move &m : legal) steps.push_back(Step{m, !turn});
        return {std::move(steps), std::move(priors), value};
    }

    bool reverse_q(const ArcRefNode<Step> &node) const override { return node->step.color == Color::Black; }  // torch.rs:49-52
};

// ---- the same backend for many games on one engine: one sc_evaluator shared by the game threads, one root slot per
// game.  The slot follows the real game (set_search_root once per real move) and `predict` passes only the moves below
// the search root; the device generates the legal moves and applies the terminal rule.
class ChessB200Slot : public Game<BoardState> {
    sc_evaluator *ev_;
    int slot_;
    size_t root_plies_ = 0;  // moves of the game stored in the slot
    bool rooted_ = false;

public:
    ChessB200Slot(sc_evaluator *ev, int slot) : ev_(ev), slot_(slot)
    {
        if (!ev) throw std::runtime_error("ChessB200Slot: null evaluator");
    }

    // the slot follows the game to `state`, the next search root: the moves played since the last call are appended
    void set_search_root(const BoardState &state)
    {
        const std::vector<Move> &ms = state.move_stack();
        if (ms.size() < root_plies_) throw std::runtime_error("set_search_root: the game is shorter than the slot's");
        std::vector<sc_move> mv;
        for (size_t k = root_plies_; k < ms.size(); k++) mv.push_back(sc_move{ms[k].from, ms[k].to, ms[k].promo, 0});
        const int rc = rooted_ ? sc_evaluator_extend_root(ev_, slot_, mv.data(), (int)mv.size())
                               : sc_evaluator_set_root(ev_, slot_, mv.data(), (int)mv.size());
        if (rc != SC_OK) throw std::runtime_error(sc_last_error());
        root_plies_ = ms.size();
        rooted_ = true;
    }

    std::tuple<std::vector<Step>, std::vector<float>, float> predict(const ArcRefNode<Step> &node, const BoardState &state,
                                                                      bool argmax) const override
    {
        if (argmax) throw std::runtime_error("predict: argmax is not used by mcts and not implemented");
        const std::vector<Move> &ms = state.move_stack();
        if (!rooted_ || ms.size() < root_plies_) throw std::runtime_error("predict: the state is not below the search root");
        int n_hist = 0;  // as ChessB200's
        for (ArcRefNode<Step> n = node; n && n_hist < SC_LOOKBACK;) {
            n_hist++;
            if (!n->parent) break;
            n = n->parent->lock();
        }
        if (n_hist > (int)ms.size() + 1) throw std::runtime_error("predict: history longer than the move stack");
        std::vector<sc_move> path;
        for (size_t k = root_plies_; k < ms.size(); k++) path.push_back(sc_move{ms[k].from, ms[k].to, ms[k].promo, 0});
        sc_move moves[SC_MAX_MOVES];
        float priors[SC_MAX_MOVES];
        int32_t cnt = 0;
        float value = 0.f;
        if (sc_evaluator_predict(ev_, slot_, path.data(), (int)path.size(), n_hist, nullptr, moves, &cnt, priors, &value) !=
            SC_OK)
            throw std::runtime_error(sc_last_error());
        if (cnt == 0) return {{}, {}, value};  // terminal: the device's torch.rs:98-106 value
        const Color turn = node->step.color;
        if (turn != state.turn()) throw std::runtime_error("predict: node and state disagree on the side to move");
        std::vector<Step> steps;
        steps.reserve((size_t)cnt);
        for (int i = 0; i < cnt; i++) steps.push_back(Step{Move{moves[i].from, moves[i].to, moves[i].promo}, !turn});
        return {std::move(steps), std::vector<float>(priors, priors + cnt), value};
    }

    bool reverse_q(const ArcRefNode<Step> &node) const override { return node->step.color == Color::Black; }
};

// ---- src/mcts.rs:61-328 ----------------------------------------------------------------------------
namespace mcts {

inline float uct(float sqrt_total_num_vis, float prior, float move_q, int32_t move_n_act, bool reverse_q, float cpuct)
{
    const float average_award = move_q / ((float)move_n_act + 1e-4f) * (reverse_q ? -1.f : 1.f);
    const float exploration = (sqrt_total_num_vis + 0.01f) / (1.f + (float)move_n_act) * cpuct * prior;
    return average_award + exploration;
}

// Iterator::max_by keeps the LAST of equal maxima; non-finite input is an error
inline std::optional<size_t> find_max(const std::vector<float> &v)
{
    if (v.empty()) return std::nullopt;
    size_t best = 0;
    for (size_t i = 0; i < v.size(); i++) {
        if (!std::isfinite(v[i])) throw std::runtime_error("!!!! CHECK the values.");
        if (v[i] >= v[best]) best = i;
    }
    return best;
}

template <class T> void backward(const std::deque<ArcRefNode<T>> &path, float reward)
{
    for (const auto &node : path) {
        node->num_act += 1;
        node->q_value += reward;
    }
}

// Dirichlet(0.3) sample of the given size; None below two moves (src/mcts.rs:123-130)
using NoiseFn = std::optional<std::vector<float>> (*)(size_t size, void *ctx);

template <class G, class S>
std::tuple<std::deque<ArcRefNode<typename S::Step>>, std::vector<typename S::Step>, float>
select(const G &game, const ArcRefNode<typename S::Step> &node, S &state, float cpuct, float epsilon, bool with_noise,
       NoiseFn get_noise = nullptr, void *noise_ctx = nullptr)
{
    using StepT = typename S::Step;
    std::deque<ArcRefNode<StepT>> path{node};
    for (;;) {
        const ArcRefNode<StepT> recent_node = path.back();
        const size_t path_len = path.size();
        auto [steps, prior, outcome] = game.predict(recent_node, state, false);
        const bool reverse_q = game.reverse_q(recent_node);
        const auto &children = recent_node->children;
        if (children.empty() || steps.empty()) return {std::move(path), std::move(steps), outcome};

        ArcRefNode<StepT> best_child;
        if (children.size() == 1)
            best_child = children[0];
        else {
            const bool is_root = path_len == 1;
            std::vector<float> prior_rand = prior;
            if (is_root && with_noise && get_noise) {
                if (auto noise = get_noise(steps.size(), noise_ctx))
                    for (size_t i = 0; i < prior_rand.size(); i++)
                        prior_rand[i] = prior[i] * (1.0f - epsilon) + (*noise)[i] * epsilon;
            }
            int32_t total = 0;
            for (const auto &c : children) total += c->num_act;
            const float sqrt_total_num_vis = std::sqrt((float)total);
            if (prior_rand.size() != children.size()) throw std::runtime_error("!!!! CHECK the values.");
            std::vector<float> uct_children(children.size());
            for (size_t i = 0; i < children.size(); i++)
                uct_children[i] =
                    uct(sqrt_total_num_vis, prior_rand[i], children[i]->q_value, children[i]->num_act, reverse_q, cpuct);
            const size_t idx = *find_max(uct_children);
            for (size_t i = 0; i < children.size(); i++) children[i]->uct = uct_children[i];
            best_child = children[idx];
        }
        state.advance(best_child->step);
        path.push_back(best_child);
    }
}

template <class G, class S>
void mcts(const G &game, const ArcRefNode<typename S::Step> &node, const S &state, int n_rollout, std::optional<float> cpuct,
          float epsilon, bool with_noise, NoiseFn get_noise = nullptr, void *noise_ctx = nullptr)
{
    using StepT = typename S::Step;
    const float c = cpuct.value_or(1.2f);
    for (int r = 0; r < n_rollout; r++) {
        S local_state = state.dup();
        auto [path, steps, reward] = select<G, S>(game, node, local_state, c, epsilon, with_noise, get_noise, noise_ctx);
        const ArcRefNode<StepT> &cur = path.back();
        const uint32_t depth = cur->depth;
        std::vector<ArcRefNode<StepT>> children;
        children.reserve(steps.size());
        for (auto &s : steps) {
            auto ch = std::make_shared<Node<StepT>>();
            ch->step = s;
            ch->depth = depth + 1;
            ch->parent = WeakRefNode<StepT>(cur);
            children.push_back(std::move(ch));
        }
        cur->children = std::move(children);
        backward(path, reward);
    }
}

// `uniform` in [0,1) drives the temperature sampling (thread_rng in the reference)
template <class S>
std::optional<typename S::Step> step(Cursor<typename S::Step> &cursor, S &state, float temp, double (*uniform)(void *) = nullptr,
                                     void *rng_ctx = nullptr)
{
    const auto &children = cursor.current().children;
    if (children.empty()) return std::nullopt;
    size_t choice = 0;
    if (temp == 0.0f) {
        for (size_t i = 1; i < children.size(); i++)
            if (children[i]->num_act > children[choice]->num_act) choice = i;  // position() of the first maximum
    } else {
        if (!uniform) throw std::runtime_error("step: temperature sampling needs a random source");
        const float power = 1.0f / temp;
        std::vector<double> w(children.size());
        double tot = 0.0;
        for (size_t i = 0; i < children.size(); i++) tot += (w[i] = std::pow((float)children[i]->num_act, power));
        const double r = uniform(rng_ctx) * tot;
        double acc = 0.0;
        choice = children.size() - 1;
        for (size_t i = 0; i < children.size(); i++) {
            acc += w[i];
            if (r < acc) {
                choice = i;
                break;
            }
        }
    }
    cursor.navigate_down(choice);
    cursor.current_mut().reset();
    const typename S::Step s = cursor.current().step;
    state.advance(s);
    return s;
}

}  // namespace mcts
}  // namespace smartchess
