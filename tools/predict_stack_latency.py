"""sc_predict_stack (leaves given as move stacks, replayed and packed on the device) against sc_predict (leaves packed on
the host) on the same games.

The bench.py net (19 blocks, seed 0).  The leaves are the positions after 40, 150 and 300 plies of seeded random games;
sc_predict gets them as the host rules pack them (sc_rules_probe) with python-chess ep_square, sc_predict_stack as move
stacks.  Per round the two calls alternate, each for --iters calls per size:
  * call time (host buffers in, host buffers out, the call returns after the results are in them) at n = 1 / 8 / 64 for
    each stack length;
  * leaf evals/s at n = 2048 for each stack length.
Then, in a pass of its own with event timing on, the replay kernel's device time at each size.  Before timing, the two
calls' outputs are checked for bit equality.  Records the card name and power limit, prints one JSON line and writes it
to --out.

    python tools/predict_stack_latency.py --out profiles/predict_stack_latency.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "smart-chess-rust_b200"))

import numpy as np  # noqa: E402

import scb200  # noqa: E402
from bench import make_blob  # noqa: E402

SIZES = (1, 8, 64, 2048)
PLIES = (40, 150, 300)
N_GAMES = 64


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def random_games(n_games, plies, seed):
    """n_games seeded uniform random games that last at least `plies` plies (move lists)"""
    rng = np.random.RandomState(seed)
    games = []
    while len(games) < n_games:
        hist = []
        for _ in range(plies):
            mv = scb200.rules_probe(hist)[0]
            if len(mv) == 0:
                break
            hist.append(tuple(int(x) for x in mv[rng.randint(len(mv))]))
        if len(hist) == plies:
            games.append(hist)
    return games


def leaves(games, plies, n):
    """n leaves (the games repeated) after `plies` plies: move stacks, and the host's packed leaves with ep_square"""
    stacks = [games[i % len(games)][:plies] for i in range(n)]
    pos = np.zeros(n, dtype=scb200.POSITION_DTYPE)
    ep = np.full(n, -1, dtype=np.int8)
    for i in range(min(n, len(games))):
        s = stacks[i]
        pos[i] = scb200.rules_probe(s)[1]
        f, t, _ = s[-1]
        if (int(pos[i]["slot"][0][0]) >> t) & 1 and abs(t - f) == 16:
            ep[i] = (f + t) // 2
    for i in range(len(games), n):
        pos[i], ep[i] = pos[i % len(games)], ep[i % len(games)]
    off = np.zeros(n + 1, dtype=np.int32)
    off[1:] = np.cumsum([len(s) for s in stacks])
    flat = np.zeros(int(off[-1]), dtype=scb200.MOVE_DTYPE)
    for s, o in zip(stacks, off[:-1]):
        for k, m in enumerate(s):
            flat[o + k] = (m[0], m[1], m[2], 0)
    return (flat, off), pos, ep


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=200, help="calls per leg at n <= 64 (a tenth of it at 2048)")
    ap.add_argument("--mode", default="bf16", choices=("bf16", "fp16", "fp32", "ffma"))
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    mode = {"bf16": scb200.SC_MODE_BF16, "fp16": scb200.SC_MODE_FP16, "fp32": scb200.SC_MODE_FP32,
            "ffma": scb200.SC_MODE_FP32_FFMA}[a.mode]
    tmp = tempfile.mkdtemp()
    _, blob = make_blob(tmp)
    games = random_games(N_GAMES, max(PLIES), seed=0)
    data = {p: leaves(games, p, SIZES[-1]) for p in PLIES}
    e = scb200.Engine(blob, 0, mode, SIZES[-1])
    n_max = SIZES[-1]
    out = (np.zeros((n_max, scb200.SC_MAX_MOVES), scb200.MOVE_DTYPE), np.zeros(n_max, np.int32),
           np.zeros((n_max, scb200.SC_MAX_MOVES), np.float32), np.zeros(n_max, np.float32))

    def sub(stk, n):
        flat, off = stk
        return flat[: off[n]], off[: n + 1]

    for p, (stk, pos, ep) in data.items():
        for n in SIZES:
            x = [np.copy(v) for v in e.predict(pos[:n], ep[:n])]
            y = e.predict_stack(sub(stk, n), positions=True)
            assert np.array_equal(x[1], y[1]) and np.array_equal(x[3].view(np.uint32), y[3].view(np.uint32)), (p, n)
            for i in range(n):  # the entries past each leaf's count are unspecified
                c = int(x[1][i])
                assert np.array_equal(x[0][i, :c].view(np.uint32), y[0][i, :c].view(np.uint32)), (p, n, i)
                assert np.array_equal(x[2][i, :c].view(np.uint32), y[2][i, :c].view(np.uint32)), (p, n, i)
            assert y[4][: min(n, N_GAMES)].tobytes() == pos[: min(n, N_GAMES)].tobytes(), (p, n)

    def call(kind, p, n):
        stk, pos, ep = data[p]
        if kind == "predict":
            e.predict(pos[:n], ep[:n], out=out)
        else:
            e.predict_stack(sub(stk, n), out=out)

    kinds = ("predict", "predict_stack")
    legs = {k: {(p, n): [] for p in PLIES for n in SIZES} for k in kinds}
    for p in PLIES:  # warm up every shape
        for n in SIZES:
            for kind in kinds:
                for _ in range(5):
                    call(kind, p, n)
    for r in range(a.rounds):
        for p in PLIES:
            for n in SIZES:
                iters = a.iters if n <= 64 else max(3, a.iters // 10)
                for kind in (kinds if r % 2 == 0 else kinds[::-1]):
                    t0 = time.perf_counter()
                    for _ in range(iters):
                        call(kind, p, n)
                    legs[kind][(p, n)].append((time.perf_counter() - t0) / iters)
    e.set_timing(1)
    replay_ms = {}
    for p in PLIES:
        for n in SIZES:
            t = []
            for _ in range(50):
                call("predict_stack", p, n)
                t.append(e.predict_stack_timing())
            replay_ms[f"plies{p}_n{n}"] = round(statistics.median(t), 4)
    e.set_timing(0)
    e.close()

    res = {"card": card(), "mode": a.mode, "rounds": a.rounds, "replay_kernel_ms_median": replay_ms}
    for kind, by in legs.items():
        r = {}
        for p in PLIES:
            for n in SIZES[:-1]:
                ms = [x * 1e3 for x in by[(p, n)]]
                r[f"call_ms_plies{p}_n{n}"] = {"median": round(statistics.median(ms), 4), "min": round(min(ms), 4),
                                              "max": round(max(ms), 4)}
            rate = [n_max / x for x in by[(p, n_max)]]
            r[f"leaf_evals_per_s_plies{p}_n2048"] = {"median": round(statistics.median(rate)), "min": round(min(rate)),
                                                     "max": round(max(rate))}
        res[kind] = r
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
