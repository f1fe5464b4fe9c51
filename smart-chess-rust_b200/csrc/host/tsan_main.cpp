// ThreadSanitizer harness for the host-side search (`make -C smart-chess-rust_b200/csrc tsan`).
//
// The reference marks its tree `unsafe impl Send` (src/mcts.rs:26) and never runs it on more than one thread; the
// batched driver walks thousands of trees with a worker pool (csrc/host/search.cpp), so the sharing discipline is
// checked here: self-play and arena runs with the stand-in (position-hash) evaluator, 8 worker threads, under TSAN.
// The batching evaluator (host/evaluator.cpp) is checked the same way: 64 game threads of sc_game_selfplay_many share
// one stand-in evaluator, and every trace must equal the same seed's game played alone.
// The engine entry points search.cpp and the evaluator link against are stubbed -- no GPU and no CUDA call is involved.
#include <cstdio>
#include <cstring>
#include <string>

#include <atomic>
#include <chrono>
#include <thread>
#include <vector>

#include "../common.cuh"
#include "evaluator.hpp"

namespace scb {
static thread_local std::string g_err;
void set_error(const std::string &msg) { g_err = msg; }
int engine_backend_create(sc_engine *, int, int *, EvalBackend **) { return SC_E_NOGPU; }
}  // namespace scb

extern "C" {
const char *sc_last_error(void) { return scb::g_err.c_str(); }
int sc_eval(sc_engine *, int, const sc_position *, const sc_move *, const int32_t *, float *, float *, void *) { return SC_E_NOGPU; }
int sc_eval_submit(sc_engine *, int, const sc_position *, const sc_move *, const int32_t *, float *, float *, void *, int *)
{
    return SC_E_NOGPU;
}
int sc_eval_wait(sc_engine *, int) { return SC_E_NOGPU; }
int sc_info(const sc_engine *, int *, int *, int *) { return SC_E_NOGPU; }
int sc_device_info(const sc_engine *, int *, int *) { return SC_E_NOGPU; }
}

static int run(bool arena, int threads, int leaves_per_tree)
{
    sc_selfplay_config cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.n_trees = 96;
    cfg.rollout_num = 24;
    cfg.num_steps = 40;
    cfg.cpuct = 2.5f;
    cfg.epsilon = 0.15f;
    cfg.with_noise = 1;
    cfg.temperature_switch = 6;
    cfg.seed = 9;
    cfg.n_threads = threads;
    cfg.evaluator = 1;
    cfg.pipeline_groups = 2;
    cfg.keep_traces = 1;
    cfg.leaves_per_tree = leaves_per_tree;
    sc_selfplay *sp = nullptr;
    int rc = arena ? sc_arena_create(nullptr, nullptr, &cfg, &sp) : sc_selfplay_create(nullptr, &cfg, &sp);
    if (rc != SC_OK) {
        fprintf(stderr, "create failed: %s\n", sc_last_error());
        return 1;
    }
    sc_selfplay_stats st;
    rc = sc_selfplay_run(sp, 192, 0, 0.0, &st);
    printf("%s threads=%d leaves_per_tree=%d: rc=%d games=%lld plies=%lld rollouts=%lld\n", arena ? "arena" : "selfplay", threads,
           leaves_per_tree, rc, (long long)st.games_finished, (long long)st.moves, (long long)st.rollouts);
    const bool ok = rc == SC_OK && st.games_finished == 192 && sc_selfplay_trace_json(sp, 191, nullptr, 0) > 0;
    sc_selfplay_destroy(sp);
    return ok ? 0 : 1;
}

// 64 games through one stand-in evaluator against the same seeds played one at a time
static int run_many()
{
    sc_selfplay_config cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.rollout_num = 12;
    cfg.num_steps = 30;
    cfg.cpuct = 2.5f;
    cfg.epsilon = 0.15f;
    cfg.with_noise = 1;
    cfg.temperature_switch = 6;
    cfg.evaluator = 1;
    const int n = 64;
    const int64_t cap = 1 << 18;
    std::vector<uint64_t> seeds(n);
    for (int g = 0; g < n; g++) seeds[g] = 1000 + 7 * g;
    std::vector<char> buf((size_t)n * cap);
    std::vector<int64_t> sizes(n);
    sc_evaluator_counts c;
    int rc = sc_game_selfplay_many(nullptr, &cfg, n, seeds.data(), buf.data(), cap, sizes.data(), &c);
    int same = 0;
    std::vector<char> one(cap);
    for (int g = 0; rc == SC_OK && g < n; g++) {
        cfg.seed = seeds[g];
        const int64_t k = sc_game_selfplay(nullptr, &cfg, one.data(), cap);
        same += k == sizes[g] && k <= cap && strcmp(one.data(), buf.data() + (size_t)g * cap) == 0;
    }
    printf("game_selfplay_many games=%d: rc=%d traces equal to the games played alone: %d; passes=%lld leaves=%lld "
           "largest batch=%lld root updates=%lld\n",
           n, rc, same, (long long)c.passes, (long long)c.leaves, (long long)c.largest_batch, (long long)c.root_updates);
    return rc == SC_OK && same == n && c.largest_batch > 1 ? 0 : 1;
}

// a backend whose first pass waits until `release` is set
struct StallingBackend : scb::EvalBackend {
    std::atomic<bool> in_pass{false}, release{false};
    void update_roots(const std::vector<scb::RootUpdate *> &) override {}
    void predict(const std::vector<scb::LeafRequest *> &r) override
    {
        in_pass = true;
        while (!release) std::this_thread::sleep_for(std::chrono::milliseconds(1));
        for (scb::LeafRequest *q : r) *q->move_cnt_out = 1;
    }
};

// destroy while one caller's pass runs and eight more callers are queued behind it: the pass completes normally, the
// queued callers get SC_E_STATE
static int run_destroy()
{
    StallingBackend *be = new StallingBackend();
    sc_evaluator *ev = nullptr;
    scb::evaluator_create(be, 16, 16, &ev);
    std::vector<int> rc(9, 1), cnt(9, 0);
    auto call = [&](int t) {
        sc_move mv[SC_MAX_MOVES];
        float pri[SC_MAX_MOVES], v;
        rc[t] = sc_evaluator_predict(ev, t, nullptr, 0, 0, nullptr, mv, &cnt[t], pri, &v);
    };
    std::vector<std::thread> th;
    th.emplace_back(call, 0);
    while (!be->in_pass) std::this_thread::sleep_for(std::chrono::milliseconds(1));
    for (int t = 1; t < 9; t++) th.emplace_back(call, t);
    std::this_thread::sleep_for(std::chrono::milliseconds(200));  // the eight callers reach the queue
    std::thread destroyer([&] { sc_evaluator_destroy(ev); });
    std::this_thread::sleep_for(std::chrono::milliseconds(50));
    be->release = true;
    destroyer.join();
    for (std::thread &t : th) t.join();
    int state = 0;
    for (int t = 1; t < 9; t++) state += rc[t] == SC_E_STATE;
    printf("evaluator destroy: running caller rc=%d count=%d, queued callers failed with SC_E_STATE: %d of 8\n", rc[0],
           cnt[0], state);
    return rc[0] == SC_OK && cnt[0] == 1 && state == 8 ? 0 : 1;
}

int main(int argc, char **argv)
{
    int bad = 0;
    if (argc > 1) {  // `prof`: one single-threaded self-play run (the gprof target of `make hostprof`)
        bad = run(false, 1, 1);
        printf(bad ? "FAILED\n" : "host profile run ok\n");
        return bad;
    }
    bad += run(false, 8, 1);
    bad += run(false, 8, 4);
    bad += run(true, 8, 1);
    bad += run_many();
    bad += run_destroy();
    printf(bad ? "FAILED\n" : "tsan harness ok\n");
    return bad;
}
