"""sc_predict_path (a stored root plus the leaf's path, replayed on the device) against sc_predict_stack (the whole game
replayed per leaf) and sc_predict (leaves packed on the host) on the same leaves.

The bench.py net (19 blocks, seed 0).  The leaves are seeded random games after R + P plies, for roots of R = 40, 150
and 300 plies and paths of P = 0, 8 and 24 plies; sc_predict_path gets root R of the game (stored by sc_set_roots) and
the P moves after it, sc_predict_stack the R + P moves, sc_predict the leaf as the host rules pack it (sc_rules_probe)
with python-chess ep_square.  Per round, for each size, with the three calls in alternating order:
  * sc_set_roots time for 1 root and for 2048 roots of R plies (host clock; the call is synchronous);
  * one-leaf call time (host buffers in, host buffers out, the call returns after the results are in them);
  * leaf evals/s at n = 2048, sc_predict_path with 2048 roots (one per leaf) and with 16 roots (128 leaves each).
Then, in a pass of its own with event timing on, the path-replay and replay kernels' device times.  Before timing, the
outputs of the three calls are checked for bit equality.  Records the card name and power limit, prints one JSON line
and writes it to --out.

    python tools/predict_path_latency.py --out profiles/predict_path_latency.json
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

ROOT_PLIES = (40, 150, 300)
PATH_PLIES = (0, 8, 24)
N = 2048
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


def host_packed(games, plies):
    """the host's packed leaves of the games after `plies` plies, with ep_square, repeated to N leaves"""
    pos = np.zeros(N, dtype=scb200.POSITION_DTYPE)
    ep = np.full(N, -1, dtype=np.int8)
    for i, g in enumerate(games):
        s = g[:plies]
        pos[i] = scb200.rules_probe(s)[1]
        f, t, _ = s[-1]
        if (int(pos[i]["slot"][0][0]) >> t) & 1 and abs(t - f) == 16:
            ep[i] = (f + t) // 2
    for i in range(len(games), N):
        pos[i], ep[i] = pos[i % len(games)], ep[i % len(games)]
    return pos, ep


def flat(lists):
    off = np.zeros(len(lists) + 1, dtype=np.int32)
    off[1:] = np.cumsum([len(s) for s in lists])
    out = np.zeros(int(off[-1]), dtype=scb200.MOVE_DTYPE)
    for s, o in zip(lists, off[:-1]):
        for k, m in enumerate(s):
            out[o + k] = (m[0], m[1], m[2], 0)
    return out, off


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=200, help="calls per one-leaf leg (a tenth of it at n = 2048)")
    ap.add_argument("--mode", default="bf16", choices=("bf16", "fp16", "fp32", "ffma"))
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    mode = {"bf16": scb200.SC_MODE_BF16, "fp16": scb200.SC_MODE_FP16, "fp32": scb200.SC_MODE_FP32,
            "ffma": scb200.SC_MODE_FP32_FFMA}[a.mode]
    tmp = tempfile.mkdtemp()
    _, blob = make_blob(tmp)
    games = random_games(N_GAMES, max(ROOT_PLIES) + max(PATH_PLIES), seed=0)
    e = scb200.Engine(blob, 0, mode, N)
    out = (np.zeros((N, scb200.SC_MAX_MOVES), scb200.MOVE_DTYPE), np.zeros(N, np.int32),
           np.zeros((N, scb200.SC_MAX_MOVES), np.float32), np.zeros(N, np.float32))

    # per (R, P): the roots (one per leaf: root i = game i % N_GAMES after R plies), the paths of the leaves over 2048
    # and over 16 roots, the whole stacks and the host-packed leaves
    roots = {r: flat([games[i % N_GAMES][:r] for i in range(N)]) for r in ROOT_PLIES}
    data = {}
    for r in ROOT_PLIES:
        for p in PATH_PLIES:
            paths = flat([games[i % N_GAMES][r : r + p] for i in range(N)])
            paths16 = flat([games[i % 16][r : r + p] for i in range(N)])
            stacks = flat([games[i % N_GAMES][: r + p] for i in range(N)])
            data[(r, p)] = (paths, paths16, stacks) + host_packed(games, r + p)
    leaf_root = np.arange(N, dtype=np.int32)
    leaf_root16 = leaf_root % 16

    def sub(lists, n):
        f, off = lists
        return f[: off[n]], off[: n + 1]

    def call(kind, r, p, n, roots16=False):
        paths, paths16, stacks, pos, ep = data[(r, p)]
        if kind == "predict":
            e.predict(pos[:n], ep[:n], out=out)
        elif kind == "predict_stack":
            e.predict_stack(sub(stacks, n), out=out)
        elif roots16:
            e.predict_path(leaf_root16[:n], sub(paths16, n), out=out)
        else:
            e.predict_path(leaf_root[:n], sub(paths, n), out=out)

    def same(x, y, what):
        assert np.array_equal(x[1], y[1]) and np.array_equal(x[3].view(np.uint32), y[3].view(np.uint32)), what
        for i in range(N):  # the entries past each leaf's count are unspecified
            c = int(x[1][i])
            assert np.array_equal(x[0][i, :c].view(np.uint32), y[0][i, :c].view(np.uint32)), (what, i)
            assert np.array_equal(x[2][i, :c].view(np.uint32), y[2][i, :c].view(np.uint32)), (what, i)

    for r in ROOT_PLIES:
        e.set_roots(roots[r])
        for p in PATH_PLIES:
            paths, paths16, stacks, pos, ep = data[(r, p)]
            x = [np.copy(v) for v in e.predict(pos, ep)]
            y = [np.copy(v) for v in e.predict_stack(stacks, positions=True)]
            same(x, y, ("predict_stack", r, p))
            assert y[4][:N_GAMES].tobytes() == pos[:N_GAMES].tobytes(), (r, p)
            z = e.predict_path(leaf_root, paths, positions=True)
            same(y, z, ("predict_path", r, p))
            assert z[4].tobytes() == y[4].tobytes(), (r, p)
            # the 16-root leaves are games 0..15 only: against predict_stack on the same games
            y = [np.copy(v) for v in e.predict_stack(flat([games[i % 16][: r + p] for i in range(N)]), positions=True)]
            z = e.predict_path(leaf_root16, paths16, positions=True)
            same(y, z, ("predict_path 16 roots", r, p))
            assert z[4].tobytes() == y[4].tobytes(), (r, p)

    kinds = ("predict", "predict_stack", "predict_path")
    legs = {}

    def leg(key, fn, iters):
        t0 = time.perf_counter()
        for _ in range(iters):
            fn()
        legs.setdefault(key, []).append((time.perf_counter() - t0) / iters)

    one_root = {r: sub(roots[r], 1) for r in ROOT_PLIES}
    for warm in (True, False):  # one pass to warm up every shape, then the timed rounds
        for rnd in range(1 if warm else a.rounds):
            it = 3 if warm else a.iters
            it_big = 2 if warm else max(3, a.iters // 10)
            for r in ROOT_PLIES:
                leg(("set_roots_1", r), lambda: e.set_roots(one_root[r]), it)
                leg(("set_roots_2048", r), lambda: e.set_roots(roots[r]), it_big)
                for p in PATH_PLIES:
                    order = kinds if rnd % 2 == 0 else kinds[::-1]
                    for kind in order:
                        leg((kind, r, p, 1), lambda: call(kind, r, p, 1), it)
                    for kind in order:
                        leg((kind, r, p, N), lambda: call(kind, r, p, N), it_big)
                    leg(("predict_path_16roots", r, p, N), lambda: call("predict_path", r, p, N, True), it_big)
        if warm:
            legs.clear()

    e.set_timing(1)
    kernel_ms = {}
    for r in ROOT_PLIES:
        e.set_roots(roots[r])
        for p in PATH_PLIES:
            for n in (1, N):
                for kind, timing in (("predict_path", e.predict_path_timing), ("predict_stack", e.predict_stack_timing)):
                    t = []
                    for _ in range(50):
                        call(kind, r, p, n)
                        t.append(timing())
                    kernel_ms[f"{kind}_roots{r}_path{p}_n{n}"] = round(statistics.median(t), 4)
    e.set_timing(0)
    e.close()

    def stat(v, scale, digits):
        v = [x * scale for x in v]
        return {"median": round(statistics.median(v), digits), "min": round(min(v), digits), "max": round(max(v), digits)}

    res = {"card": card(), "mode": a.mode, "rounds": a.rounds, "iters": a.iters,
           "replay_kernel_ms_median": kernel_ms,
           "set_roots_ms": {f"{k[0]}_roots{k[1]}": stat(v, 1e3, 4) for k, v in legs.items() if k[0].startswith("set_")}}
    for kind in kinds + ("predict_path_16roots",):
        rr = {}
        for r in ROOT_PLIES:
            for p in PATH_PLIES:
                if (kind, r, p, 1) in legs:
                    rr[f"call_ms_roots{r}_path{p}_n1"] = stat(legs[(kind, r, p, 1)], 1e3, 4)
                rr[f"leaf_evals_per_s_roots{r}_path{p}_n{N}"] = stat([1 / x for x in legs[(kind, r, p, N)]], N, 0)
        res[kind] = rr
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
