"""scb200 -- Python face of the B200 leaf-evaluation backend (libscb200.so, C ABI in
include/sc_b200.h).  Plumbing for tests and bench.py; the product is the shared library.

There is NO CPU fallback: importing works anywhere (so the symbol-table test can run on a
CPU box), but creating an Engine without an sm_100 device raises.
"""
from .binding import (  # noqa: F401
    Engine,
    Evaluator,
    EvalCacheCounts,
    SelfPlay,
    Arena,
    elo,
    rules_probe,
    rules_perft,
    game_selfplay,
    game_selfplay_many,
    last_error,
    random_positions,
    SCError,
    SC_MODE_BF16,
    SC_MODE_FP32,
    SC_MODE_FP32_FFMA,
    SC_MODE_FP16,
    SC_MODE_FP8,
    SC_MAX_MOVES,
    SC_MAX_STACK,
    SC_MAX_CACHE_ENTRIES,
    POSITION_DTYPE,
    MOVE_DTYPE,
    lib_path,
    load_library,
    pack_positions,
    DECLARED_SYMBOLS,
)
from .export import write_blob, export_checkpoint  # noqa: F401
from .random_init import random_init_state_dict  # noqa: F401
