// sc_evaluator: the queue, the dispatcher thread and the C ABI of include/sc_b200.h's batching evaluator, and the
// position-hash stand-in backend.  The device work is the backend's (host/evaluator.hpp).
#include <chrono>
#include <condition_variable>
#include <cstring>
#include <deque>
#include <memory>
#include <mutex>
#include <set>
#include <thread>

#include "../common.cuh"
#include "evaluator.hpp"
#include "host_util.hpp"

using namespace scb;

namespace {

// a request and its caller's wake-up
template <class R> struct Waiting : R {
    std::condition_variable cv;
    bool done = false;
};
using Leaf = Waiting<LeafRequest>;
using Update = Waiting<RootUpdate>;

using Clock = std::chrono::steady_clock;

}  // namespace

struct sc_evaluator {
    std::unique_ptr<EvalBackend> be;
    int n_slots = 0, max_batch = 0;
    std::mutex mu;
    std::condition_variable work;  // the dispatcher: requests are pending, or closing
    std::condition_variable left;  // sc_evaluator_destroy: no caller is blocked any more
    std::deque<Leaf *> leaves;
    std::deque<Update *> updates;
    bool closing = false;
    int callers = 0;  // blocked in a call
    sc_evaluator_counts counts{};
    std::thread dispatcher;

    void dispatch();
};

// Takes every pending update (one per slot: a second one for the same slot waits for the next pass) and up to
// max_batch pending leaves, applies the updates, then evaluates the leaves; requests that arrive meanwhile wait for the
// next pass.  On closing, fails what is still pending.
void sc_evaluator::dispatch()
{
    std::unique_lock<std::mutex> lk(mu);
    std::vector<Update *> ups;
    std::vector<Leaf *> batch;
    std::vector<RootUpdate *> up_req;
    std::vector<LeafRequest *> leaf_req;
    for (;;) {
        work.wait(lk, [&] { return closing || !leaves.empty() || !updates.empty(); });
        if (closing) break;
        ups.clear();
        batch.clear();
        std::set<int> slots;
        for (auto it = updates.begin(); it != updates.end();) {
            if (slots.insert((*it)->slot).second) {
                ups.push_back(*it);
                it = updates.erase(it);
            } else {
                ++it;
            }
        }
        while (!leaves.empty() && (int)batch.size() < max_batch) {
            batch.push_back(leaves.front());
            leaves.pop_front();
        }
        lk.unlock();
        up_req.assign(ups.begin(), ups.end());
        leaf_req.assign(batch.begin(), batch.end());
        if (!up_req.empty()) be->update_roots(up_req);
        if (!leaf_req.empty()) be->predict(leaf_req);
        lk.lock();
        counts.root_updates += (int64_t)ups.size();
        if (!batch.empty()) {
            counts.passes += 1;
            counts.leaves += (int64_t)batch.size();
            if ((int64_t)batch.size() > counts.largest_batch) counts.largest_batch = (int64_t)batch.size();
        }
        for (Update *u : ups) {
            u->done = true;
            u->cv.notify_one();
        }
        for (Leaf *q : batch) {
            q->done = true;
            q->cv.notify_one();
        }
    }
    auto fail = [](auto *r) {
        r->rc = SC_E_STATE;
        r->err = "the evaluator was destroyed before the request ran";
        r->done = true;
        r->cv.notify_one();
    };
    for (Update *u : updates) fail(u);
    for (Leaf *q : leaves) fail(q);
    updates.clear();
    leaves.clear();
}

namespace {

// queues r, blocks until the dispatcher is done with it and returns its status (its message to this thread's
// sc_last_error); the seconds it took are added to *waited (a field of ev, under its lock)
template <class R> int submit(sc_evaluator *ev, R &r, std::deque<R *> &q, const char *what, double *waited)
{
    std::unique_lock<std::mutex> lk(ev->mu);
    if (ev->closing) {
        lk.unlock();
        set_error(std::string(what) + ": the evaluator is being destroyed");
        return SC_E_STATE;
    }
    const Clock::time_point t0 = Clock::now();
    ev->callers++;
    q.push_back(&r);
    ev->work.notify_one();
    r.cv.wait(lk, [&] { return r.done; });
    if (waited && !ev->closing) *waited += std::chrono::duration<double>(Clock::now() - t0).count();
    if (--ev->callers == 0 && ev->closing) ev->left.notify_all();
    lk.unlock();  // ev may be gone from here on
    if (r.rc != SC_OK) set_error(r.err.compare(0, strlen(what), what) == 0 ? r.err : std::string(what) + ": " + r.err);
    return r.rc;
}

int update_root(sc_evaluator *ev, int slot, const sc_move *moves, int len, bool append)
{
    const char *what = append ? "sc_evaluator_extend_root" : "sc_evaluator_set_root";
    if (!ev || slot < 0 || slot >= ev->n_slots || len < 0 || (len > 0 && !moves)) {
        set_error(std::string(what) + ": bad argument" +
                  (ev && (slot < 0 || slot >= ev->n_slots)
                       ? " (slot " + std::to_string(slot) + " is not in 0.." + std::to_string(ev->n_slots - 1) + ")"
                       : ""));
        return SC_E_INVAL;
    }
    Update u;
    u.slot = slot;
    u.append = append;
    u.moves = moves;
    u.len = len;
    return submit(ev, u, ev->updates, what, nullptr);
}

// the stand-in: each slot's game on the host, host::hash_eval for priors and value.  Replays without the device's
// move checks (the callers are the search, which plays legal moves)
class HashBackend : public EvalBackend {
    std::vector<std::unique_ptr<chess::Game>> root_;

public:
    explicit HashBackend(int n_slots) : root_((size_t)n_slots) {}

    void update_roots(const std::vector<RootUpdate *> &u) override
    {
        for (RootUpdate *r : u) {
            std::unique_ptr<chess::Game> &g = root_[r->slot];
            if (r->append && !g) {
                r->rc = SC_E_STATE;
                r->err = "slot " + std::to_string(r->slot) + " has no root";
                continue;
            }
            if (!r->append) g.reset(new chess::Game());
            for (int k = 0; k < r->len; k++) g->push(chess::Move{r->moves[k].from, r->moves[k].to, r->moves[k].promo});
        }
    }

    void predict(const std::vector<LeafRequest *> &req) override
    {
        for (LeafRequest *q : req) {
            if (!root_[q->slot]) {
                q->rc = SC_E_STATE;
                q->err = "slot " + std::to_string(q->slot) + " has no root";
                continue;
            }
            chess::Game g = *root_[q->slot];
            for (int k = 0; k < q->len; k++) g.push(chess::Move{q->path[k].from, q->path[k].to, q->path[k].promo});
            chess::MoveList l;
            g.cur.legal_moves(l);
            *q->move_cnt_out = l.n;
            for (int k = 0; k < l.n; k++) q->moves_out[k] = sc_move{l.m[k].from, l.m[k].to, l.m[k].promo, 0};
            if (l.n == 0)
                *q->value_out = g.cur.in_check() ? (g.cur.turn == chess::WHITE ? -1.f : 1.f) : 0.f;
            else
                *q->value_out = host::hash_eval(g.cur, l.m, l.n, q->priors_out);
            if (q->pos_out) {
                const int plies = (int)g.moves.size();
                host::pack_position(g, q->n_hist ? q->n_hist : std::min(SC_LOOKBACK, plies + 1), q->pos_out);
            }
        }
    }
};

}  // namespace

namespace scb {

EvalBackend *hash_backend_create(int n_slots) { return new HashBackend(n_slots); }

int evaluator_create(EvalBackend *be, int n_slots, int max_batch, sc_evaluator **out)
{
    std::unique_ptr<EvalBackend> owned(be);
    sc_evaluator *ev = new sc_evaluator();
    ev->be = std::move(owned);
    ev->n_slots = n_slots;
    ev->max_batch = max_batch;
    ev->dispatcher = std::thread([ev] { ev->dispatch(); });
    *out = ev;
    return SC_OK;
}

}  // namespace scb

extern "C" {

int sc_evaluator_create(sc_engine *e, int n_slots, sc_evaluator **out)
{
    if (!out) {
        set_error("sc_evaluator_create: bad argument");
        return SC_E_INVAL;
    }
    *out = nullptr;
    EvalBackend *be = nullptr;
    int max_batch = 0;
    SCB_CHECK(engine_backend_create(e, n_slots, &max_batch, &be));
    return evaluator_create(be, n_slots, max_batch, out);
}

int sc_evaluator_destroy(sc_evaluator *ev)
{
    if (!ev) return SC_OK;
    {
        std::lock_guard<std::mutex> lk(ev->mu);
        ev->closing = true;
        ev->work.notify_all();
    }
    ev->dispatcher.join();  // completes a running pass and fails the pending requests
    {
        std::unique_lock<std::mutex> lk(ev->mu);
        ev->left.wait(lk, [&] { return ev->callers == 0; });
    }
    delete ev;  // the backend gives the engine back
    return SC_OK;
}

int sc_evaluator_set_root(sc_evaluator *ev, int slot, const sc_move *stack, int len)
{
    return update_root(ev, slot, stack, len, false);
}

int sc_evaluator_extend_root(sc_evaluator *ev, int slot, const sc_move *moves, int len)
{
    return update_root(ev, slot, moves, len, true);
}

int sc_evaluator_predict(sc_evaluator *ev, int slot, const sc_move *path, int len, int n_hist, sc_position *pos_out,
                         sc_move *moves_out, int32_t *move_cnt_out, float *priors_out, float *value_out)
{
    if (!ev || slot < 0 || slot >= ev->n_slots || len < 0 || (len > 0 && !path) || !moves_out || !move_cnt_out ||
        !priors_out || !value_out) {
        set_error(std::string("sc_evaluator_predict: bad argument") +
                  (ev && (slot < 0 || slot >= ev->n_slots)
                       ? " (slot " + std::to_string(slot) + " is not in 0.." + std::to_string(ev->n_slots - 1) + ")"
                       : ""));
        return SC_E_INVAL;
    }
    Leaf q;
    q.slot = slot;
    q.path = path;
    q.len = len;
    q.n_hist = n_hist;
    q.pos_out = pos_out;
    q.moves_out = moves_out;
    q.move_cnt_out = move_cnt_out;
    q.priors_out = priors_out;
    q.value_out = value_out;
    return submit(ev, q, ev->leaves, "sc_evaluator_predict", &ev->counts.wait_seconds);
}

int sc_evaluator_stats(sc_evaluator *ev, sc_evaluator_counts *out)
{
    if (!ev || !out) {
        set_error("sc_evaluator_stats: bad argument");
        return SC_E_INVAL;
    }
    std::lock_guard<std::mutex> lk(ev->mu);
    *out = ev->counts;
    return SC_OK;
}

}  // extern "C"
