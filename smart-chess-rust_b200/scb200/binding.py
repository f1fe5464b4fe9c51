"""ctypes binding of include/sc_b200.h."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

SC_MODE_FP32 = 0
SC_MODE_BF16 = 1
SC_MODE_FP32_FFMA = 2
SC_MODE_FP16 = 3
SC_MODE_FP8 = 4
SC_N_PLANES = 112
SC_N_META = 7
SC_N_POLICY = 4672
SC_MAX_MOVES = 256
SC_MAX_STACK = 1024

# struct sc_position { uint64_t slot[8][8]; int32_t meta[7]; int32_t n_hist; }  (544 bytes)
POSITION_DTYPE = np.dtype([("slot", np.uint64, (8, 8)), ("meta", np.int32, (7,)), ("n_hist", np.int32)])
# struct sc_move { uint8_t from, to, promo, pad; }
MOVE_DTYPE = np.dtype([("from", np.uint8), ("to", np.uint8), ("promo", np.uint8), ("pad", np.uint8)])
assert POSITION_DTYPE.itemsize == 544 and MOVE_DTYPE.itemsize == 4

DECLARED_SYMBOLS = [
    "sc_create", "sc_destroy", "sc_last_error", "sc_info", "sc_eval", "sc_eval_device", "sc_encode_only",
    "sc_move_index_only", "sc_forward_only", "sc_launch_count", "sc_last_timing", "sc_set_timing", "sc_kernel_timing",
    "sc_eval_submit", "sc_eval_wait", "sc_selfplay_create", "sc_selfplay_run", "sc_selfplay_trace_json",
    "sc_selfplay_destroy", "sc_rules_probe", "sc_arena_create", "sc_encode_steps", "sc_timed_flops_per_leaf",
    "sc_random_positions", "sc_test_dirichlet", "sc_game_selfplay", "sc_rules_perft", "sc_device_info",
    "sc_selfplay_run_many", "sc_debug_tower", "sc_rules_probe_fen", "sc_selfplay_trace_game", "sc_predict",
    "sc_predict_timing", "sc_predict_stack", "sc_predict_stack_timing", "sc_set_roots", "sc_predict_path",
    "sc_predict_path_timing", "sc_evaluator_create", "sc_evaluator_destroy", "sc_evaluator_set_root",
    "sc_evaluator_extend_root", "sc_evaluator_predict", "sc_evaluator_stats", "sc_game_selfplay_many",
]


class SelfPlayConfig(C.Structure):
    """struct sc_selfplay_config (field names follow the reference CLI, src/main.rs:25-60)"""
    _fields_ = [("n_trees", C.c_int32), ("rollout_num", C.c_int32), ("num_steps", C.c_int32), ("cpuct", C.c_float),
                ("epsilon", C.c_float), ("with_noise", C.c_int32), ("temperature_switch", C.c_int32),
                ("temperature", C.c_float), ("seed", C.c_uint64), ("n_threads", C.c_int32), ("evaluator", C.c_int32),
                ("pipeline_groups", C.c_int32), ("keep_traces", C.c_int32),
                ("leaves_per_tree", C.c_int32), ("rollout_factor", C.c_float)]


class EvaluatorCounts(C.Structure):
    """struct sc_evaluator_counts"""
    _fields_ = [("passes", C.c_int64), ("leaves", C.c_int64), ("largest_batch", C.c_int64),
                ("root_updates", C.c_int64), ("wait_seconds", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class SelfPlayStats(C.Structure):
    _fields_ = [("leaf_evals", C.c_int64), ("terminal_evals", C.c_int64), ("rollouts", C.c_int64), ("moves", C.c_int64),
                ("games_finished", C.c_int64), ("white_wins", C.c_int64), ("black_wins", C.c_int64),
                ("draws", C.c_int64), ("unfinished", C.c_int64), ("batches", C.c_int64), ("seconds", C.c_double),
                ("wait_seconds", C.c_double), ("games_dropped", C.c_int64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


_LIB = None


class SCError(RuntimeError):
    pass


def lib_path() -> str:
    return os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "libscb200.so")


def load_library():
    """Loads libscb200.so; raises loudly if the CUDA extension has not been built."""
    global _LIB
    if _LIB is None:
        p = lib_path()
        if not os.path.exists(p):
            raise SCError(f"{p} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback for this backend)")
        L = C.CDLL(p)
        L.sc_last_error.restype = C.c_char_p
        L.sc_create.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.sc_destroy.argtypes = [C.c_void_p]
        L.sc_info.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.sc_device_info.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.sc_selfplay_run_many.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int64, C.c_int64, C.c_double,
                                           C.POINTER(SelfPlayStats)]
        L.sc_debug_tower.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sc_eval.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 6
        L.sc_predict.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 7
        L.sc_predict_timing.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        L.sc_predict_stack.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 9
        L.sc_predict_stack_timing.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        L.sc_set_roots.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.sc_predict_path.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 10
        L.sc_predict_path_timing.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        # (ctypes.CDLL releases the GIL around every call: evaluator callers on Python threads overlap)
        L.sc_evaluator_create.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]
        L.sc_evaluator_destroy.argtypes = [C.c_void_p]
        L.sc_evaluator_set_root.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        L.sc_evaluator_extend_root.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        L.sc_evaluator_predict.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 5
        L.sc_evaluator_stats.argtypes = [C.c_void_p, C.POINTER(EvaluatorCounts)]
        L.sc_game_selfplay_many.argtypes = [C.c_void_p, C.POINTER(SelfPlayConfig), C.c_int, C.c_void_p, C.c_char_p,
                                            C.c_int64, C.c_void_p, C.POINTER(EvaluatorCounts)]
        L.sc_eval_device.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                     C.c_void_p, C.c_void_p]
        L.sc_encode_only.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sc_move_index_only.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sc_forward_only.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sc_encode_steps.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 4 + [C.c_int] + [C.c_void_p] * 5
        L.sc_timed_flops_per_leaf.restype = C.c_double
        L.sc_timed_flops_per_leaf.argtypes = [C.c_void_p]
        L.sc_launch_count.restype = C.c_int64
        L.sc_launch_count.argtypes = [C.c_void_p]
        L.sc_last_timing.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float)]
        L.sc_set_timing.argtypes = [C.c_void_p, C.c_int]
        L.sc_kernel_timing.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int)]
        L.sc_eval_submit.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 6 + [C.POINTER(C.c_int)]
        L.sc_eval_wait.argtypes = [C.c_void_p, C.c_int]
        L.sc_selfplay_create.argtypes = [C.c_void_p, C.POINTER(SelfPlayConfig), C.POINTER(C.c_void_p)]
        L.sc_selfplay_run.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_double, C.POINTER(SelfPlayStats)]
        L.sc_game_selfplay.restype = C.c_int64
        L.sc_game_selfplay.argtypes = [C.c_void_p, C.c_void_p, C.c_char_p, C.c_int64]
        L.sc_selfplay_trace_json.restype = C.c_int64
        L.sc_selfplay_trace_json.argtypes = [C.c_void_p, C.c_int64, C.c_char_p, C.c_int64]
        L.sc_selfplay_trace_game.restype = C.c_int64
        L.sc_selfplay_trace_game.argtypes = [C.c_void_p, C.c_int64]
        L.sc_selfplay_destroy.argtypes = [C.c_void_p]
        L.sc_arena_create.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(SelfPlayConfig), C.POINTER(C.c_void_p)]
        L.sc_random_positions.argtypes = [C.c_int, C.c_uint64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.sc_test_dirichlet.argtypes = [C.c_uint64, C.c_float, C.c_int, C.c_void_p]
        L.sc_rules_perft.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_uint64)]
        L.sc_rules_probe.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_int), C.c_void_p,
                                     C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.sc_rules_probe_fen.argtypes = [C.c_char_p] + L.sc_rules_probe.argtypes
        _LIB = L
    return _LIB


def _check(rc: int, what: str):
    if rc != 0:
        raise SCError(f"{what} failed ({rc}): {load_library().sc_last_error().decode()}")


def pack_positions(slots, metas, n_hists) -> np.ndarray:
    """Builds an sc_position array from per-leaf (slot[8,8] u64, meta[7] i32, n_hist)."""
    n = len(metas)
    out = np.zeros(n, dtype=POSITION_DTYPE)
    for i in range(n):
        out["slot"][i] = slots[i]
        out["meta"][i] = metas[i]
        out["n_hist"][i] = n_hists[i]
    return out


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, int):
        return a
    if hasattr(a, "data_ptr"):  # torch tensor (device or pinned host)
        return a.data_ptr()
    return a.ctypes.data


def _move_lists(lists, what):
    """(flat MOVE_DTYPE array, int32 offsets[n + 1]) of per-leaf move lists ((from, to, promo) tuples or MOVE_DTYPE
    arrays), or of such a pair given as it is"""
    if isinstance(lists, tuple):
        flat, off = lists
        flat = np.ascontiguousarray(flat, dtype=MOVE_DTYPE)
        off = np.ascontiguousarray(off, dtype=np.int32)
    else:
        lens = [len(st) for st in lists]
        off = np.zeros(len(lists) + 1, dtype=np.int32)
        off[1:] = np.cumsum(lens)
        flat = np.zeros(int(off[-1]), dtype=MOVE_DTYPE)
        for st, b, ln in zip(lists, off[:-1], lens):
            if ln:
                a = np.asarray(st)
                if a.dtype == MOVE_DTYPE:
                    flat[b : b + ln] = a
                else:
                    a = a.reshape(ln, -1)
                    for k, f in enumerate(("from", "to", "promo")):
                        flat[f][b : b + ln] = a[:, k]
    if len(off) < 1:
        raise SCError(f"{what}: offsets must hold n + 1 entries")
    return flat, off


def _n_hist_arg(n_hist, n, what):
    if n_hist is None:
        return None
    nh = np.asarray(n_hist)
    if len(nh) != n or nh.min(initial=1) < -128 or nh.max(initial=1) > 127:
        raise SCError(f"{what}: n_hist must hold one history length per leaf")
    return np.ascontiguousarray(nh, dtype=np.int8)


def _predict_out(out, n, what):
    """predict()'s (moves, counts, priors, values) for n leaves: new arrays, or the first n rows of `out`'s"""
    if out is None:
        out = (np.zeros((n, SC_MAX_MOVES), dtype=MOVE_DTYPE), np.zeros(n, dtype=np.int32),
               np.zeros((n, SC_MAX_MOVES), dtype=np.float32), np.zeros(n, dtype=np.float32))
    for a, dt, shape in zip(out, (MOVE_DTYPE, np.int32, np.float32, np.float32), ((SC_MAX_MOVES,), (), (SC_MAX_MOVES,), ())):
        if a.dtype != dt or a.shape[1:] != shape or len(a) < n or not a.flags.c_contiguous:
            raise SCError(f"{what}: `out` must be (moves, counts, priors, values) arrays as predict() returns them")
    return tuple(a[:n] for a in out)


class Engine:
    """`ChessTS` / `ChessOnnx` counterpart (src/backends/torch.rs:14-17, onnx.rs:8-11): owns the
    model for the lifetime of the process and evaluates batches of leaves."""

    def __init__(self, blob_path: str, device: int = 0, mode: int = SC_MODE_BF16, max_batch: int = 2048):
        L = load_library()
        h = C.c_void_p()
        _check(L.sc_create(blob_path.encode(), device, mode, max_batch, C.byref(h)), "sc_create")
        self._h = h
        self.mode = mode
        self.max_batch = max_batch
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            load_library().sc_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    def info(self):
        a, b, c, d, s = C.c_int(), C.c_int(), C.c_int(), C.c_int(), C.c_int()
        _check(load_library().sc_info(self._h, C.byref(a), C.byref(b), C.byref(c)), "sc_info")
        _check(load_library().sc_device_info(self._h, C.byref(d), C.byref(s)), "sc_device_info")
        return {"n_res_blocks": a.value, "max_batch": b.value, "mode": c.value, "device": d.value, "num_sms": s.value}

    def eval(self, positions: np.ndarray, moves: np.ndarray, move_off: np.ndarray, priors_out=None, value_out=None,
             stream: int = 0):
        """`predict` for n leaves: returns (priors CSR float32, values float32[n])."""
        n = len(positions)
        # numpy inputs are coerced to the ABI's element types (an int64 move_off or a strided view would otherwise be
        # reinterpreted) unless they already have them; torch tensors (pinned host buffers of bench.py) are taken as they are
        def _as(a, dt):
            if hasattr(a, "data_ptr") or (a.dtype == dt and a.flags.c_contiguous):
                return a
            return np.ascontiguousarray(a, dtype=dt)

        positions, moves, move_off = _as(positions, POSITION_DTYPE), _as(moves, MOVE_DTYPE), _as(move_off, np.int32)
        total = int(move_off[n]) if n else 0
        if priors_out is None:
            priors_out = np.zeros(max(total, 1), dtype=np.float32)
        if value_out is None:
            value_out = np.zeros(max(n, 1), dtype=np.float32)
        _check(load_library().sc_eval(self._h, n, _ptr(positions), _ptr(moves), _ptr(move_off), _ptr(priors_out),
                                      _ptr(value_out), stream or None), "sc_eval")
        return priors_out[:total], value_out[:n]

    def predict(self, positions: np.ndarray, ep_square=None, out=None, stream: int = 0, check: bool = True):
        """`Game::predict` for n leaves (sc_predict): legal moves generated on the device, then the network.
        ep_square: python-chess `ep_square` per leaf (-1 for none), or None for -1 everywhere.  Returns
        (moves MOVE_DTYPE[n, 256], counts int32[n], priors float32[n, 256], values float32[n]); leaf i's moves and priors
        are the first counts[i] entries of row i, and a leaf with counts[i] == 0 is terminal (value -1 / +1 for the
        mated side to move White / Black, 0 for stalemate).  `out`: these four arrays to fill instead of new ones (at
        least n rows each).  check=False returns the outputs with the status code (rc, moves, counts, priors, values)
        instead of raising."""
        n = len(positions)
        positions = np.ascontiguousarray(positions, dtype=POSITION_DTYPE)
        if ep_square is not None:
            ep = np.asarray(ep_square)
            if len(ep) != n or ep.min(initial=-1) < -128 or ep.max(initial=-1) > 127:
                raise SCError("predict: ep_square must hold one square (or -1) per leaf")
            ep_square = np.ascontiguousarray(ep, dtype=np.int8)
        moves, counts, priors, values = _predict_out(out, n, "predict")
        rc = load_library().sc_predict(self._h, n, _ptr(positions), _ptr(ep_square), _ptr(moves), _ptr(counts),
                                       _ptr(priors), _ptr(values), stream or None)
        if not check:
            return rc, moves, counts, priors, values
        _check(rc, "sc_predict")
        return moves, counts, priors, values

    def predict_stack(self, stacks, n_hist=None, out=None, positions: bool = False, stream: int = 0, check: bool = True):
        """predict() for leaves given as move stacks (sc_predict_stack): the device replays each game from the initial
        position and packs the leaf itself.  stacks: a list of per-leaf move lists ((from, to, promo) tuples or
        MOVE_DTYPE arrays; python-chess `board.move_stack`, oldest first, castling as the king's two-square move), or
        (flat MOVE_DTYPE array, int32 offsets[n + 1]).  n_hist: per-leaf history slots (1..8, at most plies + 1), or
        None for min(8, plies + 1).  Returns predict()'s (moves, counts, priors, values), then the packed leaves
        (POSITION_DTYPE[n]) when `positions`; check=False puts the status code first instead of raising."""
        return self._predict_moves(None, stacks, n_hist, out, positions, stream, check)

    def set_roots(self, stacks):
        """Stores root games on the device for predict_path() (sc_set_roots): stacks as predict_stack()'s.  Replaces
        the previous roots; an empty list clears them."""
        flat, off = _move_lists(stacks, "set_roots")
        _check(load_library().sc_set_roots(self._h, len(off) - 1, _ptr(flat) if len(flat) else None, _ptr(off)),
               "sc_set_roots")

    def predict_path(self, root, paths, n_hist=None, out=None, positions: bool = False, stream: int = 0,
                     check: bool = True):
        """predict_stack() for leaves given as a stored root (an index into set_roots()' list) and the moves played
        after it (sc_predict_path): leaf i is root[i]'s game followed by paths[i].  paths as predict_stack()'s stacks;
        n_hist and the result as predict_stack()'s for the whole game."""
        return self._predict_moves(np.asarray(root), paths, n_hist, out, positions, stream, check)

    def _predict_moves(self, root, lists, n_hist, out, positions, stream, check):
        """predict_stack() (root None) and predict_path() (root: its root argument as an array)"""
        what = "predict_stack" if root is None else "predict_path"
        flat, off = _move_lists(lists, what)
        n = len(off) - 1
        fn, lead = load_library().sc_predict_stack, ()
        if root is not None:
            if root.shape != (n,) or root.min(initial=0) < -2**31 or root.max(initial=0) >= 2**31:
                raise SCError("predict_path: root must hold one root index per leaf")
            root = np.ascontiguousarray(root, dtype=np.int32)
            fn, lead = load_library().sc_predict_path, (_ptr(root),)
        n_hist = _n_hist_arg(n_hist, n, what)
        moves, counts, priors, values = _predict_out(out, n, what)
        pos = np.zeros(n, dtype=POSITION_DTYPE) if positions else None
        rc = fn(self._h, n, *lead, _ptr(flat) if len(flat) else None, _ptr(off), _ptr(n_hist), _ptr(pos), _ptr(moves),
                _ptr(counts), _ptr(priors), _ptr(values), stream or None)
        res = (moves, counts, priors, values) + ((pos,) if positions else ())
        if not check:
            return (rc,) + res
        _check(rc, "sc_" + what)
        return res

    def predict_path_timing(self) -> float:
        """device time (ms) of the path-replay kernel of the last predict_path() (timing level >= 1)"""
        ms = C.c_float()
        _check(load_library().sc_predict_path_timing(self._h, C.byref(ms)), "sc_predict_path_timing")
        return ms.value

    def predict_stack_timing(self) -> float:
        """device time (ms) of the replay kernel of the last predict_stack() (timing level >= 1)"""
        ms = C.c_float()
        _check(load_library().sc_predict_stack_timing(self._h, C.byref(ms)), "sc_predict_stack_timing")
        return ms.value

    def predict_timing(self) -> float:
        """device time (ms) of the legal-move kernel of the last predict() (timing level >= 1)"""
        ms = C.c_float()
        _check(load_library().sc_predict_timing(self._h, C.byref(ms)), "sc_predict_timing")
        return ms.value

    def eval_device(self, n, d_pos, d_moves, d_off, n_moves_total, d_priors, d_value, stream: int = 0):
        _check(load_library().sc_eval_device(self._h, n, _ptr(d_pos), _ptr(d_moves), _ptr(d_off), n_moves_total,
                                             _ptr(d_priors), _ptr(d_value), stream or None), "sc_eval_device")

    def submit(self, positions, moves_strided, move_cnt, priors_out_strided, value_out, stream: int = 0) -> int:
        """Asynchronous `predict` (sc_eval_submit): moves / priors strided by 256 per leaf, buffers must stay alive
        (and should be pinned) until `wait(ticket)` returns.  At most SC_MAX_INFLIGHT = 4 tickets in flight."""
        t = C.c_int(-1)
        _check(load_library().sc_eval_submit(self._h, len(positions), _ptr(positions), _ptr(moves_strided), _ptr(move_cnt),
                                             _ptr(priors_out_strided), _ptr(value_out), stream or None, C.byref(t)),
               "sc_eval_submit")
        return t.value

    def wait(self, ticket: int):
        _check(load_library().sc_eval_wait(self._h, ticket), "sc_eval_wait")

    def encode_only(self, positions: np.ndarray):
        n = len(positions)
        positions = np.ascontiguousarray(positions, dtype=POSITION_DTYPE)
        planes = np.zeros((n, 8, 8, SC_N_PLANES), dtype=np.int8)
        meta = np.zeros((n, SC_N_META), dtype=np.int32)
        _check(load_library().sc_encode_only(self._h, n, _ptr(positions), _ptr(planes), _ptr(meta)), "sc_encode_only")
        return planes, meta

    def move_index_only(self, positions: np.ndarray, moves: np.ndarray, move_off: np.ndarray):
        n = len(positions)
        positions = np.ascontiguousarray(positions, dtype=POSITION_DTYPE)
        moves = np.ascontiguousarray(moves, dtype=MOVE_DTYPE)
        move_off = np.ascontiguousarray(move_off, dtype=np.int32)
        out = np.full(int(move_off[n]) if n else 0, -7, dtype=np.int32)
        _check(load_library().sc_move_index_only(self._h, n, _ptr(positions), _ptr(moves), _ptr(move_off), _ptr(out)),
               "sc_move_index_only")
        return out

    def forward_only(self, planes: np.ndarray, meta: np.ndarray):
        """planes float32 [n,112,8,8], meta float32 [n,7] -> (logp [n,4672], value [n])."""
        planes = np.ascontiguousarray(planes, dtype=np.float32)
        meta = np.ascontiguousarray(meta, dtype=np.float32)
        n = planes.shape[0]
        logp = np.zeros((n, SC_N_POLICY), dtype=np.float32)
        value = np.zeros(n, dtype=np.float32)
        _check(load_library().sc_forward_only(self._h, n, _ptr(planes), _ptr(meta), _ptr(logp), _ptr(value)),
               "sc_forward_only")
        return logp, value

    def encode_steps(self, steps, apply_mirror: bool = False):
        """`libsmartchess.chess_encode_steps(steps, apply_mirror)` (src/lib.rs:47-128): steps is the list
        [((from, to, promo), [((from, to, promo), visit_count), ...]), ...] a trace yields (py/dataset.py:70-77).
        Returns a list of (planes int8[8,8,112], meta int32[7], dist float32[4672], [move indices])."""
        n = len(steps)
        played = np.zeros(n, dtype=MOVE_DTYPE)
        off = np.zeros(n + 1, dtype=np.int32)
        cm, cc = [], []
        for i, (mv, children) in enumerate(steps):
            played[i] = (int(mv[0]), int(mv[1]), int(mv[2]), 0)
            for m, c in children:
                cm.append((int(m[0]), int(m[1]), int(m[2]), 0))
                cc.append(int(c))
            off[i + 1] = len(cm)
        cm = np.array(cm, dtype=MOVE_DTYPE) if cm else np.zeros(1, dtype=MOVE_DTYPE)
        cc = np.array(cc, dtype=np.uint32) if cc else np.zeros(1, dtype=np.uint32)
        planes = np.zeros((n, 8, 8, SC_N_PLANES), dtype=np.int8)
        meta = np.zeros((n, SC_N_META), dtype=np.int32)
        dist = np.zeros((n, SC_N_POLICY), dtype=np.float32)
        index = np.zeros(max(1, n * 256), dtype=np.int32)
        ioff = np.zeros(n + 1, dtype=np.int32)
        _check(load_library().sc_encode_steps(self._h, n, _ptr(played), _ptr(cm), _ptr(cc), _ptr(off), int(apply_mirror),
                                              _ptr(planes), _ptr(meta), _ptr(dist), _ptr(index), _ptr(ioff)),
               "sc_encode_steps")
        return [(planes[i], meta[i], dist[i], index[ioff[i]:ioff[i + 1]].tolist()) for i in range(n)]

    def debug_tower(self, positions, n_layers: int, which: int):
        """test hook sc_debug_tower: (x, t, y) activation buffers as uint16 [n, 64, 256] after n_layers layers
        (bf16 bit patterns on a bf16 engine, fp16 on an fp16 engine, an fp8 engine's e4m3 values as fp16)"""
        n = len(positions)
        positions = np.ascontiguousarray(positions, dtype=POSITION_DTYPE)
        out = [np.zeros((n, 64, 256), dtype=np.uint16) for _ in range(3)]
        _check(load_library().sc_debug_tower(self._h, n, _ptr(positions), n_layers, which, _ptr(out[0]), _ptr(out[1]),
                                             _ptr(out[2])), "sc_debug_tower")
        return out

    def launch_count(self) -> int:
        return int(load_library().sc_launch_count(self._h))

    def set_timing(self, level: int):
        _check(load_library().sc_set_timing(self._h, int(level)), "sc_set_timing")

    def kernel_timing(self):
        """(average ms of a 3x3 tower conv launch in the last call, number of launches)"""
        a, n = C.c_float(), C.c_int()
        _check(load_library().sc_kernel_timing(self._h, C.byref(a), C.byref(n)), "sc_kernel_timing")
        return a.value, n.value

    def timed_flops_per_leaf(self) -> float:
        return float(load_library().sc_timed_flops_per_leaf(self._h))

    def last_timing(self):
        a, b = C.c_float(), C.c_float()
        _check(load_library().sc_last_timing(self._h, C.byref(a), C.byref(b)), "sc_last_timing")
        return a.value, b.value


def _one_move_list(moves, what):
    flat, _ = _move_lists([moves], what)
    return flat


class Evaluator:
    """Batching evaluator (sc_evaluator_*): many threads, each searching one game through the one-leaf interface,
    share `engine`.  Each game keeps its root in one of n_slots slots.  Every call blocks until its request ran; the
    engine refuses direct calls while the evaluator exists."""

    def __init__(self, engine, n_slots: int):
        h = C.c_void_p()
        _check(load_library().sc_evaluator_create(engine.handle, n_slots, C.byref(h)), "sc_evaluator_create")
        self._h = h
        self._engine = engine  # keep alive
        self.n_slots = n_slots

    def close(self):
        """sc_evaluator_destroy: callers blocked in predict / set_root / extend_root get SC_E_STATE, and so does every
        later call on this object"""
        if getattr(self, "_h", None):
            h, self._h = self._h, None
            load_library().sc_evaluator_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_root(self, slot: int, stack, check: bool = True):
        """stores the game `stack` (moves from the initial position, as predict_stack()'s) as slot's root"""
        return self._update(load_library().sc_evaluator_set_root, "sc_evaluator_set_root", slot, stack, check)

    def extend_root(self, slot: int, moves, check: bool = True):
        """appends `moves` to slot's stored game"""
        return self._update(load_library().sc_evaluator_extend_root, "sc_evaluator_extend_root", slot, moves, check)

    def _update(self, fn, what, slot, moves, check):
        flat = _one_move_list(moves, what)
        rc = fn(self._h, slot, _ptr(flat) if len(flat) else None, len(flat))
        if check:
            _check(rc, what)
        return rc

    def predict(self, slot: int, path, n_hist: int = 0, positions: bool = False, check: bool = True):
        """one leaf: slot's root followed by `path`.  Returns (moves MOVE_DTYPE[256], count, priors float32[256],
        value) as one row of Engine.predict_path(), then the packed leaf when `positions`; check=False puts the status
        code first instead of raising (the message is then sc_last_error() of this thread)."""
        flat = _one_move_list(path, "predict")
        h = self._h
        if h is None:
            if check:
                raise SCError("sc_evaluator_predict failed (-5): the evaluator is closed")
            return (-5, None, 0, None, 0.0) + ((None,) if positions else ())
        moves = np.zeros(SC_MAX_MOVES, dtype=MOVE_DTYPE)
        priors = np.zeros(SC_MAX_MOVES, dtype=np.float32)
        cnt, value = np.zeros(1, dtype=np.int32), np.zeros(1, dtype=np.float32)
        pos = np.zeros(1, dtype=POSITION_DTYPE) if positions else None
        rc = load_library().sc_evaluator_predict(h, slot, _ptr(flat) if len(flat) else None, len(flat), int(n_hist),
                                                 _ptr(pos), _ptr(moves), _ptr(cnt), _ptr(priors), _ptr(value))
        res = (moves, int(cnt[0]), priors, float(value[0])) + ((pos[0],) if positions else ())
        if not check:
            return (rc,) + res
        _check(rc, "sc_evaluator_predict")
        return res

    def stats(self):
        """{passes, leaves, largest_batch, root_updates, wait_seconds}"""
        c = EvaluatorCounts()
        _check(load_library().sc_evaluator_stats(self._h, C.byref(c)), "sc_evaluator_stats")
        return c.as_dict()


def last_error() -> str:
    """sc_last_error() of the calling thread"""
    return load_library().sc_last_error().decode()


def game_selfplay_many(engine, seeds, rollout_num=20, num_steps=150, cpuct=2.5, epsilon=0.15, with_noise=False,
                       temperature_switch=0, temperature=0.0, evaluator="engine", cap=1 << 18):
    """game_selfplay() for len(seeds) games at once, each on its own host thread, all through one evaluator on
    `engine` (sc_game_selfplay_many).  Returns (traces, evaluator counts)."""
    import json

    L = load_library()
    n = len(seeds)
    cfg = SelfPlayConfig(1, rollout_num, num_steps, cpuct, epsilon, int(with_noise), temperature_switch, temperature, 0,
                         1, 0 if evaluator == "engine" else 1, 1, 1, 1, 0.0)
    sd = np.ascontiguousarray(seeds, dtype=np.uint64)
    sizes = np.zeros(n, dtype=np.int64)
    buf = C.create_string_buffer(n * cap)
    counts = EvaluatorCounts()
    _check(L.sc_game_selfplay_many(engine.handle if engine is not None else None, C.byref(cfg), n, _ptr(sd), buf, cap,
                                   _ptr(sizes), C.byref(counts)), "sc_game_selfplay_many")
    if sizes.max() > cap:
        raise SCError(f"game_selfplay_many: a trace needs {int(sizes.max())} bytes, more than cap = {cap}")
    raw = buf.raw
    traces = [json.loads(raw[g * cap : g * cap + int(sizes[g]) - 1].decode()) for g in range(n)]
    return traces, counts.as_dict()


class SelfPlay:
    """Batched counterpart of the `selfplay` binary (src/main.rs:153-238): n_trees games in flight,
    one leaf per tree per device batch.  evaluator="hash" needs no engine (test hook)."""

    def __init__(self, engine, n_trees=2048, rollout_num=180, num_steps=150, cpuct=2.5, epsilon=0.15,
                 with_noise=True, temperature_switch=4, temperature=0.0, seed=0, n_threads=0, evaluator="engine",
                 pipeline_groups=2, keep_traces=False, black_engine=None, arena=False, leaves_per_tree=1,
                 rollout_factor=0.0):
        import json as _json

        self._json = _json
        L = load_library()
        cfg = SelfPlayConfig(n_trees, rollout_num, num_steps, cpuct, epsilon, int(with_noise), temperature_switch,
                             temperature, seed, n_threads, 0 if evaluator == "engine" else 1, pipeline_groups,
                             int(keep_traces), int(leaves_per_tree), float(rollout_factor))
        h = C.c_void_p()
        self._engine = (engine, black_engine)  # keep alive
        if arena:
            _check(L.sc_arena_create(engine.handle if engine is not None else None,
                                     black_engine.handle if black_engine is not None else None, C.byref(cfg),
                                     C.byref(h)), "sc_arena_create")
        else:
            _check(L.sc_selfplay_create(engine.handle if engine is not None else None, C.byref(cfg), C.byref(h)),
                   "sc_selfplay_create")
        self._h = h

    def run(self, max_games=0, max_moves=0, max_seconds=0.0):
        st = SelfPlayStats()
        _check(load_library().sc_selfplay_run(self._h, max_games, max_moves, max_seconds, C.byref(st)), "sc_selfplay_run")
        return st.as_dict()

    @staticmethod
    def run_many(drivers, max_games=0, max_moves=0, max_seconds=0.0):
        """sc_selfplay_run_many: every driver on its own host thread of this process (one engine per GPU)."""
        n = len(drivers)
        hs = (C.c_void_p * n)(*[d._h for d in drivers])
        st = (SelfPlayStats * n)()
        _check(load_library().sc_selfplay_run_many(hs, n, max_games, max_moves, max_seconds, st), "sc_selfplay_run_many")
        return [s.as_dict() for s in st]

    def trace(self, k: int):
        L = load_library()
        n = L.sc_selfplay_trace_json(self._h, k, None, 0)
        if n < 0:
            return None
        buf = C.create_string_buffer(n)
        L.sc_selfplay_trace_json(self._h, k, buf, n)
        return self._json.loads(buf.value.decode())

    def trace_game(self, k: int) -> int:
        """start order (0-based) of the game the k-th finished trace belongs to; -1 if there is no such trace"""
        return int(load_library().sc_selfplay_trace_game(self._h, k))

    def close(self):
        if getattr(self, "_h", None):
            load_library().sc_selfplay_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def game_selfplay(engine, rollout_num=20, num_steps=150, cpuct=2.5, epsilon=0.15, with_noise=False,
                  temperature_switch=0, temperature=0.0, seed=0, evaluator="engine"):
    """One game of the `selfplay` binary (src/main.rs:153-238) through the C++ mirror of the reference's
    `Game` / `mcts` interface (csrc/host/game.hpp), one leaf per `predict`.  Returns the trace dict."""
    import json

    L = load_library()
    cfg = SelfPlayConfig(1, rollout_num, num_steps, cpuct, epsilon, int(with_noise), temperature_switch, temperature, seed,
                         1, 0 if evaluator == "engine" else 1, 1, 1, 1, 0.0)
    cap = 1 << 24
    buf = C.create_string_buffer(cap)
    n = L.sc_game_selfplay(engine.handle if engine is not None else None, C.byref(cfg), buf, cap)
    if n < 0:
        raise SCError("sc_game_selfplay failed: " + L.sc_last_error().decode())
    return json.loads(buf.value.decode())


def rules_perft(fen, depth: int) -> int:
    """perft of the driver's native rules (fen None = start position)."""
    n = C.c_uint64()
    _check(load_library().sc_rules_perft(fen.encode() if fen else None, depth, C.byref(n)), "sc_rules_perft")
    return int(n.value)


def rules_probe(history, fen=None):
    """history: list of (from, to, promo) [from `fen`, default the initial position] -> (legal moves [n,3] uint8,
    sc_position record, (termination, winner))."""
    h = np.zeros(len(history), dtype=MOVE_DTYPE)
    for i, m in enumerate(history):
        h[i] = (int(m[0]), int(m[1]), int(m[2]), 0)
    legal = np.zeros(256, dtype=MOVE_DTYPE)
    n, term, win = C.c_int(), C.c_int(), C.c_int()
    pos = np.zeros(1, dtype=POSITION_DTYPE)
    _check(load_library().sc_rules_probe_fen(fen.encode() if fen else None, _ptr(h) if len(h) else None, len(h), _ptr(legal),
                                             C.byref(n), _ptr(pos), C.byref(term), C.byref(win)), "sc_rules_probe")
    mv = np.stack([legal["from"][: n.value], legal["to"][: n.value], legal["promo"][: n.value]], axis=1)
    return mv, pos[0], (term.value, win.value)


class Arena(SelfPlay):
    """`play --black-type nn` for n_trees games at once (src/play.rs:241-343): `white` moves on even plies."""

    def __init__(self, white, black, n_trees=256, rollout=100, cpuct=1.5, temperature=0.0, temperature_switch=8,
                 max_plies=200, seed=0, n_threads=0, evaluator="engine", pipeline_groups=2, keep_traces=False,
                 leaves_per_tree=1):
        super().__init__(white, n_trees=n_trees, rollout_num=rollout, num_steps=max_plies, cpuct=cpuct,
                         with_noise=False, temperature_switch=temperature_switch, temperature=temperature, seed=seed,
                         n_threads=n_threads, evaluator=evaluator, pipeline_groups=pipeline_groups,
                         keep_traces=keep_traces, black_engine=black, arena=True, leaves_per_tree=leaves_per_tree)


def elo(total: int, wins: int, losses: int) -> float:
    """scripts/elo.py:17-19: Elo difference from a Total/Win/Loss tally."""
    import math

    s = (wins + (total - wins - losses) / 2) / total
    return 400 * math.log(s / (1 - s), 10)


def random_positions(n: int, seed: int = 1, max_ply: int = 150):
    """Synthetic workload from the driver's native rules: (sc_position[n], sc_move[total], move_off[n+1])."""
    pos = np.zeros(n, dtype=POSITION_DTYPE)
    moves = np.zeros(max(1, n * 64), dtype=MOVE_DTYPE)
    off = np.zeros(n + 1, dtype=np.int32)
    _check(load_library().sc_random_positions(n, seed, max_ply, _ptr(pos), _ptr(moves), _ptr(off), len(moves)),
           "sc_random_positions")
    return pos, moves[: int(off[n])].copy(), off
