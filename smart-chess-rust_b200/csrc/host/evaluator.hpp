// The batching evaluator of include/sc_b200.h (sc_evaluator_*): host threads submit one leaf or one root update at a
// time, one dispatcher thread (host/evaluator.cpp) runs whatever is pending as one pass of a backend.  The backend is
// the engine (engine.cu: the slot table on the device, sc_predict_path's replay and launches) or the position-hash
// stand-in (host/evaluator.cpp), which needs no GPU and lets the thread-sanitizer build run the queue.
#pragma once
#include <string>
#include <vector>

#include "../../../include/sc_b200.h"

namespace scb {

// sc_evaluator_set_root (append = false) / sc_evaluator_extend_root (append = true) of `slot`
struct RootUpdate {
    int slot;
    bool append;
    const sc_move *moves;
    int len;
    int rc = SC_OK;
    std::string err;
};

// sc_evaluator_predict: the slot's root followed by path[0, len); n_hist 0 = min(SC_LOOKBACK, plies + 1)
struct LeafRequest {
    int slot;
    const sc_move *path;
    int len, n_hist;
    sc_position *pos_out;  // may be null
    sc_move *moves_out;    // SC_MAX_MOVES entries
    int32_t *move_cnt_out;
    float *priors_out;     // SC_MAX_MOVES entries
    float *value_out;
    int rc = SC_OK;
    std::string err;
};

// one pass each; a request that fails gets its own rc and err and leaves the others alone.  Called from the dispatcher
// thread only
struct EvalBackend {
    virtual ~EvalBackend() = default;
    // updates of distinct slots
    virtual void update_roots(const std::vector<RootUpdate *> &u) = 0;
    virtual void predict(const std::vector<LeafRequest *> &r) = 0;
};

// the engine's backend with n_slots root slots (engine.cu); the engine refuses direct calls until it is destroyed
int engine_backend_create(sc_engine *e, int n_slots, int *max_batch, EvalBackend **out);
// the position-hash stand-in (the batched driver's `evaluator = 1`): priors and value of host::hash_eval
EvalBackend *hash_backend_create(int n_slots);
// an evaluator around `be` (taken over, also on failure)
int evaluator_create(EvalBackend *be, int n_slots, int max_batch, sc_evaluator **out);

}  // namespace scb
