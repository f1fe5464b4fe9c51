/*
 * sc_b200.h -- C ABI of the B200 leaf-evaluation backend for smart-chess-rust.
 *
 * This is what a new `src/backends/b200.rs` would bind (see INTEGRATION.md).  Every entry
 * point names the reference interface it replaces (paths relative to the reference repo).
 * Plain pointers and sizes only; no torch types.  All functions return 0 on success or a
 * negative SC_E_* code; `sc_last_error()` gives the message.  The reference has no error
 * channel (every failure is unwrap()/panic!, e.g. src/backends/torch.rs:30-31), so the Rust
 * shim panics on a non-zero status.
 *
 * Threading: a handle is single-threaded like the reference backends (src/game.rs takes
 * &self but every backend is !Sync in practice: RefCell at src/backends/onnx.rs:9-11).
 * Use one handle per worker thread / per GPU, or share one engine between many game threads through the
 * batching evaluator below, whose calls may come from any thread.
 */
#ifndef SC_B200_H
#define SC_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SC_OK 0
#define SC_E_INVAL (-1)   /* bad argument                         */
#define SC_E_CUDA (-2)    /* CUDA runtime / driver error          */
#define SC_E_IO (-3)      /* weight blob unreadable / malformed   */
#define SC_E_NOGPU (-4)   /* no sm_100 device: there is NO CPU fallback */
#define SC_E_STATE (-5)

#define SC_MODE_FP32 0 /* parity mode (1e-4 gate): fp32 arithmetic; the 256-wide convolutions run on the tensor
                          cores as bf16x3 split operands (6 bf16 products per fp32 product) with fp32 accumulate  */
#define SC_MODE_BF16 1 /* throughput mode: tcgen05 bf16 operands, fp32 accumulate      */
#define SC_MODE_FP32_FFMA 2 /* FP32 on the CUDA cores only (FFMA): the referee of the parity mode                */
#define SC_MODE_FP16 3 /* tensor cores with fp16 operands, fp32 accumulate: the kernels and launch structure of
                          SC_MODE_BF16, rounding where it rounds but to fp16 (11 significant bits instead of 8).  A
                          parked value (a layer output, the SE input) beyond +-65504 becomes +-inf, as in the reference's
                          fp16 autocast; a weight beyond that range fails sc_create with SC_E_IO                  */
#define SC_MODE_FP8 4  /* throughput mode with fp8 (e4m3) tensor-core operands, fp32 accumulate: the weights of every
                          tensor-core layer are e4m3 with a power-of-two scale per output channel, each layer's output
                          is stored as e4m3 (round to nearest even, saturated to +-448); LayerNorm, SE, the SE weights
                          and the heads' tails stay as in SC_MODE_BF16.  Every batch size runs the throughput kernels
                          (there is no latency kernel), so a one-leaf call takes about as long as a 128-leaf one   */

#define SC_LOOKBACK 8       /* src/chess.rs:23 */
#define SC_N_PLANES 112     /* 8 x 14, py/module.py:118-121 */
#define SC_N_META 7         /* src/chess.rs:652-662 */
#define SC_N_POLICY 4672    /* 8 x 8 x 73 */
#define SC_MAX_MOVES 256

/*
 * One leaf as `_encode` (src/chess.rs:845-877) sees it: up to 8 boards of history, newest
 * first, each as python-chess bitboards (a1 = bit 0, h8 = bit 63, white-oriented, NOT
 * rotated -- the rotation of `Board::rotate`, src/chess.rs:594-621, happens on the device),
 * plus the `encode_meta` vector of the current board (src/chess.rs:652-662).
 *
 *   slot[t][0..5] = pawns, knights, bishops, rooks, queens, kings (both colours)
 *   slot[t][6]    = white occupancy
 *   slot[t][7]    = bit 0: is_repetition(2), bit 1: is_repetition(3)   (src/chess.rs:375-380)
 *   meta          = [turn(1=white), fullmove_number, K-castle(stm), Q-castle(stm),
 *                    K-castle(opp), Q-castle(opp), halfmove_clock]
 *   n_hist        = number of valid slots, 1..8 (history stops at the tree root)
 */
typedef struct sc_position {
    uint64_t slot[SC_LOOKBACK][8];
    int32_t meta[SC_N_META];
    int32_t n_hist;
} sc_position; /* 544 bytes */

/* `chess::Move` (src/chess.rs:36-41): squares are rank*8+file; promo 0 or 2..5 (N,B,R,Q). */
typedef struct sc_move {
    uint8_t from, to, promo, pad;
} sc_move;

typedef struct sc_engine sc_engine;

/* -------- lifecycle: replaces tch::CModule::load_on_device (src/main.rs:88-94,
 *          src/play.rs:356-365) / ort Session (src/main.rs:107-113) ------------------------- */
int sc_create(const char *weights_blob_path, int device, int mode, int max_batch, sc_engine **out);
int sc_destroy(sc_engine *e);
const char *sc_last_error(void);
/* number of residual blocks found in the blob; max batch; mode */
int sc_info(const sc_engine *e, int *n_res_blocks, int *max_batch, int *mode);
/* CUDA device ordinal the engine lives on and its SM count (one engine per worker thread / per GPU,
 * the in-process form of scripts/run_batch:21's one process per job) */
int sc_device_info(const sc_engine *e, int *device, int *num_sms);

/* -------- the hot path: replaces chess_tch_predict (src/backends/torch.rs:89-146) and
 *          ChessOnnx::predict (src/backends/onnx.rs:13-56) for n non-terminal leaves ---------
 * pos[n], moves = CSR over leaves (move_off[n+1]), priors_out CSR by move_off, value_out[n]
 * (White's perspective, py/module.py:147-149).  Host pointers; pinned memory makes the copies
 * asynchronous.  `stream` is a cudaStream_t (NULL = the engine's own stream); the call
 * returns after the results are in the host buffers. */
int sc_eval(sc_engine *e, int n, const sc_position *pos, const sc_move *moves, const int32_t *move_off,
            float *priors_out, float *value_out, void *stream);

/* same computation, inputs/outputs already resident in device memory, asynchronous on
 * `stream` (no host copies, no sync): the leg bench.py reports as `value`. */
int sc_eval_device(sc_engine *e, int n, const void *d_pos, const void *d_moves, const void *d_move_off,
                   int n_moves_total, void *d_priors_out, void *d_value_out, void *stream);

/* Game::predict for n leaves in one call (src/game.rs:3-15, src/backends/torch.rs:89-146): legal moves generated on the
 * device in python-chess order (the generator of the native rules), then the network.
 * ep_square[i] = python-chess `ep_square` (the skipped square after any double push) or -1; NULL = -1 for all.  Any
 * other value, or n > max_batch, fails with SC_E_INVAL.
 * moves_out / priors_out strided by SC_MAX_MOVES (as sc_eval_submit): leaf i owns [i*SC_MAX_MOVES, +move_cnt_out[i]);
 * the call copies back the whole stride, and the entries past move_cnt_out[i] are unspecified.  A leaf with
 * move_cnt_out[i] == 0 is terminal and value_out[i] is torch.rs:98-106's rule in White's perspective (the checkmated
 * side loses, stalemate 0).  A leaf with more than SC_MAX_MOVES pseudo-legal moves (not a legal position; a legal one
 * has at most 218 legal moves) fails the call with SC_E_INVAL; the outputs are still written, at most SC_MAX_MOVES
 * moves per leaf.  Host pointers, synchronous, all modes; staging and kernels as sc_eval. */
int sc_predict(sc_engine *e, int n, const sc_position *pos, const int8_t *ep_square, sc_move *moves_out,
               int32_t *move_cnt_out, float *priors_out, float *value_out, void *stream);

/* sc_predict for n leaves given as move stacks instead of packed positions: the device replays each game with the
 * native rules and packs the leaf as the batched driver does (src/chess.rs:356-412,553-591,845-877).
 * Leaf i is the initial position (`chess.Board()`, src/main.rs:155) followed by stack[stack_off[i] .. stack_off[i+1]):
 * python-chess `board.move_stack`, oldest move first, castling as the king's two-square move.
 * n_hist[i] = the history slots `_encode` sees: the node and up to 7 ancestors, stopping at the tree root
 * (src/chess.rs:851-867); 1..8 and at most the stack length + 1 (chess.rs:863).  NULL = min(8, length + 1), the game
 * root (the batched driver's pack_leaf).  Slots are newest first, each with its is_repetition(2)/(3) flags, then meta
 * (encode_meta) and python-chess `ep_square`; then the call is sc_predict on those leaves: same moves, priors, values
 * and terminal rule, all modes, synchronous, host pointers.  pos_out (may be NULL) receives the n packed leaves, for
 * sc_eval / sc_encode_only.
 * SC_E_INVAL before any launch: sc_predict's n / NULL checks, stack_off[0] != 0 or decreasing offsets, a stack longer
 * than SC_MAX_STACK, a move with from/to >= 64 or promo not in {0, 2, 3, 4, 5}, an n_hist out of range.
 * SC_E_INVAL after the outputs are written (as sc_predict's overflow; the message names the leaf and the ply): a move
 * whose from-square holds no piece of the side to move, whose to-square holds a piece of the side to move or a king,
 * that promotes anything but a pawn reaching the last rank, or a pawn reaching the last rank without a promotion; that
 * leaf is packed from the moves before it.  Legality (pins, moving into check) is not verified, as python-chess
 * Board.push does not verify it: such a leaf is packed from whatever the replay gives. */
#define SC_MAX_STACK 1024 /* plies in one leaf's move stack (sc_predict_stack) */
int sc_predict_stack(sc_engine *e, int n, const sc_move *stack, const int32_t *stack_off, const int8_t *n_hist,
                     sc_position *pos_out, sc_move *moves_out, int32_t *move_cnt_out, float *priors_out,
                     float *value_out, void *stream);

/* Stored game roots, so that a search replays its game once per real move instead of once per leaf.
 * sc_set_roots replays n_roots games (stack / stack_off as sc_predict_stack's) on the device and keeps, per root, what
 * a later sc_predict_path needs to continue it: the final position (its ep square included) and the per-ply replay
 * records.  The table replaces the previous one and lives until the next sc_set_roots or sc_destroy; n_roots = 0 clears
 * it.  0 <= n_roots <= max_batch.  Host-side argument errors as sc_predict_stack's, before any launch and with the table
 * left as it was.  A replay-time rejection returns SC_E_INVAL naming the root and the ply, and leaves the engine without
 * roots.  Synchronous, on the engine's stream; sc_predict, sc_predict_stack and sc_eval* do not touch the table. */
int sc_set_roots(sc_engine *e, int n_roots, const sc_move *stack, const int32_t *stack_off);

/* Leaf i is root[i]'s game followed by path[path_off[i] .. path_off[i+1]).  Every output (pos_out, moves, counts,
 * priors, values, terminal rule, status, error messages) is what sc_predict_stack returns for the concatenated stack
 * root ++ path, with the same n_hist meaning and limits (NULL = min(8, total length + 1)).  Plies in messages count
 * from the initial position.  SC_E_STATE if no roots are set (also for n = 0); SC_E_INVAL if root[i] is outside
 * [0, n_roots) or the total length exceeds SC_MAX_STACK, and for path_off / path / n_hist as sc_predict_stack's
 * stack_off / stack / n_hist. */
int sc_predict_path(sc_engine *e, int n, const int32_t *root, const sc_move *path, const int32_t *path_off,
                    const int8_t *n_hist, sc_position *pos_out, sc_move *moves_out, int32_t *move_cnt_out,
                    float *priors_out, float *value_out, void *stream);

/* -------- batching evaluator: many host threads, each running one game's sequential search through the one-leaf
 * interface (src/game.rs:3-15), share one engine.  Each call carries one leaf or one root update and blocks until it is
 * done; one dispatcher thread takes every request pending when the device becomes free (up to max_batch leaves),
 * applies the pending root updates in one launch, then evaluates the leaves as one sc_predict_path-style pass and wakes
 * the callers.  Requests that arrive during a pass wait for the next one, so a lone caller sees about the latency of
 * one sc_predict_path(n = 1) call and the batches grow with the number of callers.  There is no timer and no setting.
 * Every game keeps its own root slot, 0 <= slot < n_slots, in a device table of its own: sc_set_roots' table is not
 * touched.  The evaluator is the only user of the engine's stream while it lives: every other call on the engine
 * that uses the device (sc_eval*, sc_predict*, sc_set_roots, sc_encode_*, sc_forward_only, sc_debug_tower,
 * sc_set_timing, sc_destroy) returns SC_E_STATE until sc_evaluator_destroy.  All evaluator calls but create and
 * destroy may come from any thread; error messages go to the calling thread's sc_last_error. */
typedef struct sc_evaluator sc_evaluator;
/* 1 <= n_slots <= max_batch; every slot starts empty.  SC_E_STATE if the engine already has an evaluator */
int sc_evaluator_create(sc_engine *e, int n_slots, sc_evaluator **out);
/* Fails the requests still waiting with SC_E_STATE (a pass already running completes), waits until their callers have
 * returned and gives the engine back.  Not concurrent with other calls on `ev` made after it started. */
int sc_evaluator_destroy(sc_evaluator *ev);
/* Stores stack[0, len) (a game from the initial position, as sc_predict_stack's stacks) as slot's root, replayed on
 * the device; extend_root appends moves[0, len) to the slot's stored game and replays only those, from the stored
 * position.  Returns once the slot is updated; the update is ordered before every later predict on the slot.  Updates
 * of several slots pending at once share one launch, and other slots are left untouched.  SC_E_INVAL before any
 * launch and with the slot left as it was: a bad slot, len < 0, a NULL array with len > 0, a game longer than
 * SC_MAX_STACK in all, bad move fields (sc_set_roots' checks).  SC_E_STATE: extend_root of an empty slot.  A replay-time
 * rejection returns SC_E_INVAL naming the slot and the ply (counted from the initial position) and leaves the slot
 * empty. */
int sc_evaluator_set_root(sc_evaluator *ev, int slot, const sc_move *stack, int len);
int sc_evaluator_extend_root(sc_evaluator *ev, int slot, const sc_move *moves, int len);
/* One leaf: slot's root followed by path[0, len), with n_hist history slots (0 = min(8, total length + 1)).  Outputs,
 * status and messages are those of sc_predict_path for that leaf against the slot's root (moves_out / priors_out hold
 * SC_MAX_MOVES entries, the first *move_cnt_out of them valid; pos_out may be NULL), whichever other leaves share its
 * pass; the messages name the slot instead of a leaf index.  A rejected leaf fails its own call only.  SC_E_STATE: the
 * slot is empty, or the evaluator is being destroyed. */
int sc_evaluator_predict(sc_evaluator *ev, int slot, const sc_move *path, int len, int n_hist, sc_position *pos_out,
                         sc_move *moves_out, int32_t *move_cnt_out, float *priors_out, float *value_out);
typedef struct sc_evaluator_counts {
    int64_t passes;        /* dispatcher passes that evaluated leaves */
    int64_t leaves;        /* leaves evaluated (rejected ones included) */
    int64_t largest_batch; /* most leaves in one pass */
    int64_t root_updates;  /* set_root / extend_root calls applied */
    double wait_seconds;   /* summed over predict calls: time from submission to the result */
} sc_evaluator_counts;
int sc_evaluator_stats(sc_evaluator *ev, sc_evaluator_counts *out);

/* asynchronous form of sc_eval for double-buffered callers: submit returns as soon as the work is
 * queued on `stream` (host buffers must be pinned and stay untouched until the wait returns);
 * moves and priors are STRIDED: leaf i owns moves[i*SC_MAX_MOVES .. +move_cnt[i]) and the same
 * range of priors_out.  At most SC_MAX_INFLIGHT tickets may be outstanding. */
#define SC_MAX_INFLIGHT 4
int sc_eval_submit(sc_engine *e, int n, const sc_position *pos, const sc_move *moves_strided,
                   const int32_t *move_cnt, float *priors_out_strided, float *value_out, void *stream,
                   int *ticket);
int sc_eval_wait(sc_engine *e, int ticket);

/* -------- bit-exact gates ------------------------------------------------------------------ */
/* `_encode` (src/chess.rs:845-877): planes_out int8 [n][8][8][112] (rank, file, channel), the
 * `Array3<i8>` the reference builds; meta_out int32 [n][7].  Host pointers. */
int sc_encode_only(sc_engine *e, int n, const sc_position *pos, int8_t *planes_out, int32_t *meta_out);
/* `Move::rotate` + `Move::encode` (src/chess.rs:533-550, queenmoves.rs, knightmoves.rs,
 * underpromotions.rs): index_out CSR by move_off; turn comes from pos[i].meta[0]. */
int sc_move_index_only(sc_engine *e, int n, const sc_position *pos, const sc_move *moves,
                       const int32_t *move_off, int32_t *index_out);

/* -------- training-data batch encoder: `chess_encode_steps` (src/lib.rs:47-128), the call
 * py/dataset.py:47-87 makes once per trace.  The game is replayed from the start position with the
 * native rules; for every ply i the outputs are what the reference returns for that step:
 *   planes_out  int8 [n][8][8][112]   `history.view(...)` (identical with and without apply_mirror)
 *   meta_out    int32 [n][7]          `step.encode_meta()`; with apply_mirror it is the ROTATED board's
 *                                     meta (turn flipped, fullmove+1 on White's plies, castling pairs swapped)
 *   dist_out    float [n][4672]       visit counts / (sum + 1e-5) scattered at the move indices
 *   index_out   int32 CSR             move indices of the LEGAL moves in generation order; index_off[n+1]
 * `played[i]` is the move made at ply i, children (CSR by child_off) are the (move, visit count) pairs of
 * the trace row.  Like the reference (which panics) the call fails with SC_E_INVAL if the children of a
 * ply are not exactly its legal moves or the played move is not among them. n <= max_batch. */
int sc_encode_steps(sc_engine *e, int n, const sc_move *played, const sc_move *child_moves,
                    const uint32_t *child_counts, const int32_t *child_off, int apply_mirror, int8_t *planes_out,
                    int32_t *meta_out, float *dist_out, int32_t *index_out, int32_t *index_off);

/* -------- tolerance gate: ChessModule.forward (py/module.py:135-154) -------------------------
 * planes float [n][112][8][8] (NCHW, what the backends feed), meta float [n][7];
 * logp_out float [n][4672] in the reference's flatten order, value_out float [n]. Host pointers. */
int sc_forward_only(sc_engine *e, int n, const float *planes, const float *meta, float *logp_out,
                    float *value_out);

/* -------- accounting ------------------------------------------------------------------------ */
/* kernels launched by this engine since creation (bench.py's gpu_launches) */
int64_t sc_launch_count(const sc_engine *e);
/* average device time in ms of the conv tower kernels / all kernels of the most recent
 * sc_eval* call, measured with CUDA events on the launching stream (profiling aid) */
int sc_last_timing(sc_engine *e, float *tower_ms, float *total_ms);
/* per-call event timing: 0 off, 1 = tower/total of a call (two event records + one sync per
 * call), 2 = additionally one event pair around every 3x3 tower convolution launch */
int sc_set_timing(sc_engine *e, int enabled);
/* level 2: average device time (ms) of the timed tower-convolution launches of the most recent call and
 * how many there were (the roofline kernel of bench.py): one launch of the whole-tower kernel, or the 38
 * per-layer 3x3 256->256 launches with SCB200_TOWER=0; sc_timed_flops_per_leaf = algorithmic FLOPs per
 * leaf those launches cover together */
int sc_kernel_timing(sc_engine *e, float *conv3x3_avg_ms, int *n_launches);
double sc_timed_flops_per_leaf(const sc_engine *e);
/* level >= 1: device time (ms) of the legal-move kernel of the most recent sc_predict call (CUDA events on its stream) */
int sc_predict_timing(sc_engine *e, float *movegen_ms);
/* level >= 1: device time (ms) of the replay kernel of the most recent sc_predict_stack call (CUDA events on its
 * stream); sc_predict_timing reports that call's legal-move kernel */
int sc_predict_stack_timing(sc_engine *e, float *replay_ms);
/* level >= 1: device time (ms) of the path-replay kernel of the most recent sc_predict_path call */
int sc_predict_path_timing(sc_engine *e, float *replay_ms);

/* ===================== batched self-play driver (host side, C++) ================================
 * Replaces the single-tree loop of the `selfplay` binary (src/main.rs:153-238) and `mcts::mcts` /
 * `mcts::step` (src/mcts.rs:237-328) for thousands of concurrent games: every search tree keeps the
 * reference's sequential semantics (one rollout at a time per tree: select by PUCT, expand all legal
 * moves, back up the white-perspective value), and the leaves of all trees are evaluated as one
 * device batch per step.  Priors are stored on the children at expansion, which removes the
 * reference's re-evaluation of every node on each descent (src/mcts.rs:149-153) without changing
 * any result.  Field names follow the reference's CLI (src/main.rs:25-60). */
typedef struct sc_selfplay_config {
    int32_t n_trees;            /* games in flight (BASELINE configs[2]: 2048) */
    int32_t rollout_num;        /* --rollout-num; 0 together with rollout_factor 0 = the reference's default of 300 */
    int32_t num_steps;          /* --num-steps: maximum plies per game */
    float cpuct;                /* --cpuct */
    float epsilon;              /* --epsilon: Dirichlet(0.3) mix at the root (src/mcts.rs:171-184) */
    int32_t with_noise;         /* main.rs passes true; parity runs pass 0 */
    int32_t temperature_switch; /* --temperature-switch: plies played at temperature 1 */
    float temperature;          /* --temperature after the switch (0 = first max-N child) */
    uint64_t seed;              /* per-tree RNG streams derive from this */
    int32_t n_threads;          /* host worker threads walking the trees */
    int32_t evaluator;          /* 0 = the engine (GPU); 1 = position-hash stand-in (test hook, no engine) */
    int32_t pipeline_groups;    /* 1 or 2: trees are split in groups that alternate between host and device */
    int32_t keep_traces;        /* keep the traces of finished games in memory (sc_selfplay_trace_json) */
    int32_t leaves_per_tree;    /* 0/1: one leaf per tree per batch, the reference's exact sequential search.
                                   K > 1: up to K leaves per tree per batch; in-flight paths carry a virtual loss
                                   (one visit lost by the mover).  Not visit-count identical to the reference.
                                   -1: 1 while the trees fill the batch, then trees-of-the-group / trees-still-playing
                                   (<= 16) so that the tail of a finite run keeps the device busy. */
    float rollout_factor;       /* --rollout-factor (src/main.rs:175-180): > 0 (then rollout_num must be 0): the rollouts
                                   of a move are min(300, (int)(legal moves at the root * rollout_factor)) */
} sc_selfplay_config;

typedef struct sc_selfplay_stats {
    int64_t leaf_evals;     /* network-evaluated leaves */
    int64_t terminal_evals; /* rollouts that ended in a position without legal moves (no network call) */
    int64_t rollouts;
    int64_t moves;          /* plies played (search results consumed) */
    int64_t games_finished;
    int64_t white_wins, black_wins, draws, unfinished; /* unfinished = hit num_steps without an outcome */
    int64_t batches;
    double seconds;         /* wall time of sc_selfplay_run */
    double wait_seconds;    /* of which: host waiting for the device */
    int64_t games_dropped;  /* games abandoned because the network returned a non-finite prior / value for one of
                               their leaves (the reference only prints a warning, src/backends/torch.rs:129-135);
                               the slot starts the run's next game, the other games are not affected */
} sc_selfplay_stats;

typedef struct sc_selfplay sc_selfplay;

int sc_selfplay_create(sc_engine *e, const sc_selfplay_config *cfg, sc_selfplay **out);
/* plays until `max_games` games have finished (each tree slot starts a new game when one ends), or
 * until `max_moves` plies were played in total (<= 0: no limit), or `max_seconds` elapsed (<= 0: none).
 * ONE run per driver object: a second call returns SC_E_STATE (create a new driver instead). */
int sc_selfplay_run(sc_selfplay *sp, int64_t max_games, int64_t max_moves, double max_seconds,
                    sc_selfplay_stats *stats);
/* In-process multi-GPU: runs n drivers (each created on its own engine, normally one engine per GPU) on n host
 * threads of THIS process and returns when all have finished -- the in-process form of scripts/run_batch:21
 * (the reference scales by independent processes; a Rust host has no torchrun).  Every driver gets the same
 * limits; stats[i] belongs to sps[i].  Games are sharded by the caller (seeds / max_games per driver); there
 * is no exchange between the drivers.  Returns the first non-zero status. */
int sc_selfplay_run_many(sc_selfplay **sps, int n, int64_t max_games, int64_t max_moves, double max_seconds,
                         sc_selfplay_stats *stats);
/* trace of the k-th finished game in the format of src/trace.rs:23-32
 * ({"steps": [[uci, q, [[uci, n, q, uct], ...]], ...], "outcome": {...} | null}); returns the number
 * of bytes needed (including the NUL); copies at most `cap`. */
int64_t sc_selfplay_trace_json(sc_selfplay *sp, int64_t k, char *buf, int64_t cap);
/* which game the k-th finished trace is: the game's start order within the run (0-based; the games sitting in the tree
 * slots at the start are 0 .. n_trees-1, every later game takes the next number when its slot frees up); -1 if k is out
 * of range.  Lets a caller name trace files by game instead of by finishing order (scripts/run_batch: trace{k}.json). */
int64_t sc_selfplay_trace_game(sc_selfplay *sp, int64_t k);
int sc_selfplay_destroy(sc_selfplay *sp);

/* One self-play game through the one-leaf-at-a-time interface of the reference: the C++ mirror of
 * `trait Game` / `mcts::mcts` / `mcts::step` (src/game.rs:3-21, src/mcts.rs:132-328; csrc/host/game.hpp)
 * and the move loop of src/main.rs:153-238, with `predict` = sc_eval of one leaf (predict runs at every
 * level of every descent, as in the reference).  Uses rollout_num, num_steps, cpuct, epsilon, with_noise,
 * temperature_switch, temperature, seed, evaluator of `cfg`.  Writes the trace (format above) to `buf`;
 * returns the bytes needed including the NUL, or -1 (sc_last_error). */
int64_t sc_game_selfplay(sc_engine *e, const sc_selfplay_config *cfg, char *buf, int64_t cap);

/* sc_game_selfplay for n_games games at once, game i with seed seeds[i], each on its own host thread, all predicting
 * through one evaluator of n_games slots on `e` (cfg->evaluator = 0; n_games <= max_batch) or through the position-hash
 * stand-in (cfg->evaluator = 1, e unused).  Each game owns one slot: before every search it extends the slot by the
 * moves played since, and its leaves pass only the moves below the search root.  Game i's trace goes to
 * buf + i * cap (at most cap bytes with the NUL; buf may be NULL), the bytes it needs to sizes[i].  counts_out (may be
 * NULL): the evaluator's sc_evaluator_stats at the end.  Returns SC_OK, or the first game's error (sc_last_error). */
int sc_game_selfplay_many(sc_engine *e, const sc_selfplay_config *cfg, int n_games, const uint64_t *seeds, char *buf,
                          int64_t cap, int64_t *sizes, sc_evaluator_counts *counts_out);

/* ---- arena: two networks play each other (the `play` binary with --black-type nn, src/play.rs:241-343,
 * and scripts/leader-board).  Both players share one configuration, as the reference's CLI does
 * (src/play.rs:43-81): rollout_num = --rollout, cpuct, temperature, temperature_switch; noise is off
 * (play.rs:250), temperature 0 picks uniformly among the most visited children (play.rs:269-278), a game
 * ends when outcome(claim_draw=true) is set after a ply or after num_steps (200) plies.  `white` moves on
 * even plies.  Within a pipeline group every game is at a ply of the same parity (a slot whose game ended
 * starts the run's next game at the next even group ply), so each device batch belongs to one network and
 * the batches stay full.  Colour-swapped games = a second arena with the engines exchanged, as
 * scripts/leader-board:49-54 does. */
int sc_arena_create(sc_engine *white, sc_engine *black, const sc_selfplay_config *cfg, sc_selfplay **out);

/* Synthetic workload (SURVEY 8d): seeded uniform random play from the start position with the driver's
 * native rules, restart on mate/stalemate or at `max_ply`; every non-terminal position met is emitted
 * with its true history (packed leaf, node depth = ply) and its legal moves (CSR).  Fills exactly n. */
int sc_random_positions(int n, uint64_t seed, int max_ply, sc_position *pos_out, sc_move *moves_out,
                        int32_t *move_off /* n+1 */, int max_moves_total);

/* Test hook (bf16, fp16 and fp8 engines): encodes n leaves and runs only the first n_layers (0 = all 41: stem, 19 x (conv1, conv2),
 * the two 256-wide head 1x1 convolutions) of the convolution tower with the throughput kernel (which = 0) or the
 * small-batch latency kernel (which = 1, not on fp8 engines); copies the three activation buffers (bf16 / fp16 bit patterns,
 * an fp8 engine's e4m3 values as the fp16 bit patterns of the same values, [n][64][256]:
 * x = block input / output, t = conv1 output / policy head input, y = value head input) to the host.  Lets the tests
 * compare the two kernels layer by layer. */
int sc_debug_tower(sc_engine *e, int n, const sc_position *pos, int n_layers, int which, uint16_t *x_out,
                   uint16_t *t_out, uint16_t *y_out);

/* Test hook: one Dirichlet(alpha) sample of size n from the driver's root-noise sampler (src/mcts.rs:123-130
 * uses rand_distr::Dirichlet(0.3)); lets the tests check its moments. */
int sc_test_dirichlet(uint64_t seed, float alpha, int n, float *out);

/* perft (number of leaf nodes of the legal-move tree of the given depth <= 7) of the driver's native rules from a
 * FEN (NULL = start position): pins the move generator to the published perft tables. */
int sc_rules_perft(const char *fen, int depth, uint64_t *nodes);

/* Host rules probe: replays `n_history` moves from the start position with the driver's native rules
 * (the replacement of the python-chess calls at src/chess.rs:665-788) and reports what the reference
 * would see there: legal moves in python-chess generation order, the packed leaf `_encode` would be
 * given (node depth = ply), and outcome(claim_draw=True) (termination code of src/chess.rs:87-105 or
 * 0, winner 1/0/-1).  Returns SC_E_INVAL if a history move is not legal. */
int sc_rules_probe(const sc_move *history, int n_history, sc_move *legal_out, int *n_legal, sc_position *packed_out,
                   int *termination, int *winner);
/* the same from an arbitrary start position (`chess.Board(fen)`; NULL = the initial position) */
int sc_rules_probe_fen(const char *fen, const sc_move *history, int n_history, sc_move *legal_out, int *n_legal,
                       sc_position *packed_out, int *termination, int *winner);

#ifdef __cplusplus
}
#endif
#endif /* SC_B200_H */
