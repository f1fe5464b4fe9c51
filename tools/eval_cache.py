"""What the evaluation cache (sc_set_eval_cache) gains and costs, cached against uncached engines of the same blob in
the same run (the order of the two alternates).  Writes profiles/eval_cache.json (or --out).

1. One-leaf sc_predict_path calls on the 19-block seed-0 net in bf16 and fp8: a leaf seen for the first time (miss),
   the same leaf again (hit), and the same leaf on an uncached engine.  Median over --leaves distinct leaves.
2. Miss-only sc_predict calls at n = 1, 64 and 2048 (every leaf new to a fresh table): what the probe, the added wait
   and the finish kernel cost when nothing hits.  bf16.
3. Whole games through sc_game_selfplay_many at 1, 64 and 2048 games (bf16), uncached and with tables of 2^16 and 2^20
   entries, on two workloads:
   - configs[0] settings (noise off, temperature 0): every game is the same game, so the leaves of one pass repeat
     each other -- the best case for the cache;
   - diverse: root noise (epsilon 0.15), temperature 1 for the first 30 plies, a distinct seed per game.
   Per run: plies/s, hit and duplicate shares of the lookups, mean pass size, and whether every trace equals the
   uncached run's trace of the same seed.
"""
import argparse
import json
import os
import statistics
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "smart-chess-rust_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from evaluator_throughput import gpu_info  # noqa: E402


def random_games(n_games, max_plies, seed):
    import scb200

    rng = np.random.RandomState(seed)
    games = []
    for _ in range(n_games):
        hist = []
        while len(hist) < max_plies:
            mv = scb200.rules_probe(hist)[0]
            if len(mv) == 0:
                break
            hist.append(tuple(int(x) for x in mv[rng.randint(len(mv))]))
        games.append(hist)
    return games


def timed(fn):
    t0 = time.perf_counter()
    fn()
    return (time.perf_counter() - t0) * 1e3


def one_leaf(blob, mode, n_leaves, table):
    """median ms of one-leaf sc_predict_path calls: miss, hit, uncached (each leaf distinct: a prefix of a random game
    as the root and the game's next plies as the path)"""
    import scb200

    games = random_games(8, 120, seed=17)
    roots = [g[:60] for g in games]
    leaves = list(dict.fromkeys((r, tuple(g[60 : 60 + 1 + j])) for j in range(60) for r, g in enumerate(games)))
    leaves = leaves[:n_leaves]
    ref = scb200.Engine(blob, 0, mode, 64)
    e = scb200.Engine(blob, 0, mode, 64)
    e.set_eval_cache(table)
    for eng in (ref, e):
        eng.set_roots(roots)
        for _ in range(20):  # warm-up
            eng.predict_path([0], [games[0][60:61]])
    e.set_eval_cache(table)
    miss, hit, unc = [], [], []
    for k, (r, p) in enumerate(leaves):
        def call(eng):
            return lambda: eng.predict_path([r], [list(p)])
        if k % 2:
            unc.append(timed(call(ref)))
        miss.append(timed(call(e)))
        hit.append(timed(call(e)))
        if not k % 2:
            unc.append(timed(call(ref)))
    st = e.eval_cache_stats()
    ref.close()
    e.close()
    return {"mode": {scb200.SC_MODE_BF16: "bf16", scb200.SC_MODE_FP8: "fp8"}[mode], "leaves": len(leaves), "counts": st,
            "miss_ms": statistics.median(miss), "hit_ms": statistics.median(hit), "uncached_ms": statistics.median(unc),
            "hit_over_uncached": statistics.median(hit) / statistics.median(unc),
            "miss_over_uncached": statistics.median(miss) / statistics.median(unc)}


def miss_only(blob, sizes, reps, table):
    """median ms of sc_predict calls whose leaves are all new to a fresh table, and of the same calls uncached"""
    import scb200

    need = max(sizes) * reps
    pos = scb200.random_positions(3 * need, seed=23)[0]
    _, first = np.unique(pos.view(np.uint8).reshape(len(pos), -1), axis=0, return_index=True)
    pos = pos[np.sort(first)][:need]
    assert len(pos) == need
    ref = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, max(sizes))
    e = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, max(sizes))
    e.set_eval_cache(table)
    out = []
    for n in sizes:
        for eng in (ref, e):
            for _ in range(5):
                eng.predict(pos[:n])  # warm-up
        cached, unc = [], []
        for r in range(reps):
            batch = pos[r * n : (r + 1) * n]
            e.set_eval_cache(table)
            if r % 2:
                unc.append(timed(lambda: ref.predict(batch)))
            cached.append(timed(lambda: e.predict(batch)))
            if not r % 2:
                unc.append(timed(lambda: ref.predict(batch)))
            assert e.eval_cache_stats()["hits"] == 0
        out.append({"n": n, "reps": reps, "cached_ms": statistics.median(cached), "uncached_ms": statistics.median(unc),
                    "cached_over_uncached": statistics.median(cached) / statistics.median(unc)})
    ref.close()
    e.close()
    return out


def games_runs(blob, games, tables, num_steps):
    import scb200

    workloads = {
        "configs[0] (best case: every game is the same game)": dict(rollout_num=20, cpuct=2.5, seeds=lambda n: [0] * n),
        "diverse (noise on, epsilon 0.15, temperature switch 30, distinct seeds)":
            dict(rollout_num=20, cpuct=2.5, with_noise=True, epsilon=0.15, temperature_switch=30, temperature=0.0,
                 seeds=lambda n: list(range(1000, 1000 + n))),
    }
    eng = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, max(games))
    out = []
    for wname, w in workloads.items():
        kw = {k: v for k, v in w.items() if k != "seeds"}
        for n in games:
            seeds = w["seeds"](n)
            ref_traces = None
            for table in [0] + tables:
                eng.set_eval_cache(table)
                scb200.game_selfplay_many(eng, seeds[:1], num_steps=2, **kw)  # warm-up
                eng.set_eval_cache(table)
                t0 = time.perf_counter()
                traces, c = scb200.game_selfplay_many(eng, seeds, num_steps=num_steps, **kw)
                dt = time.perf_counter() - t0
                st = eng.eval_cache_stats()
                plies = sum(len(t["steps"]) for t in traces)
                if table == 0:
                    ref_traces = traces
                r = {"workload": wname, "games": n, "table": table, "seconds": dt, "plies": plies,
                     "plies_per_s": plies / dt, "leaves": c["leaves"], "passes": c["passes"],
                     "mean_batch": c["leaves"] / max(1, c["passes"]),
                     "hit_share": st["hits"] / max(1, st["lookups"]),
                     "duplicate_share": st["duplicates"] / max(1, st["lookups"]),
                     "evictions": st["evictions"], "traces_equal_uncached": traces == ref_traces}
                print(json.dumps(r), flush=True)
                out.append(r)
    eng.set_eval_cache(0)
    eng.close()
    for r in out:
        base = next(x for x in out if x["workload"] == r["workload"] and x["games"] == r["games"] and x["table"] == 0)
        r["speedup"] = r["plies_per_s"] / base["plies_per_s"]
    return out


def main():
    import scb200

    ap = argparse.ArgumentParser()
    ap.add_argument("--leaves", type=int, default=200)
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--games", default="1,64,2048")
    ap.add_argument("--tables", default="65536,1048576")
    ap.add_argument("--num-steps", type=int, default=60)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "eval_cache.json"))
    a = ap.parse_args()
    tables = [int(x) for x in a.tables.split(",")]
    res = {"net": "19-block seed-0", **gpu_info(),
           "whole_games": "rollout_num 20, cpuct 2.5, num_steps %d, bf16" % a.num_steps}
    with tempfile.TemporaryDirectory() as d:
        blob = os.path.join(d, "seed0.scw")
        scb200.write_blob(scb200.random_init_state_dict(19, 0), blob)
        res["one_leaf_predict_path"] = [one_leaf(blob, m, a.leaves, tables[0])
                                        for m in (scb200.SC_MODE_BF16, scb200.SC_MODE_FP8)]
        print(json.dumps(res["one_leaf_predict_path"]), flush=True)
        res["miss_only_predict_bf16"] = miss_only(blob, (1, 64, 2048), a.reps, tables[0])
        print(json.dumps(res["miss_only_predict_bf16"]), flush=True)
        res["selfplay_many"] = games_runs(blob, [int(x) for x in a.games.split(",")], tables, a.num_steps)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
