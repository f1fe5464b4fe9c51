"""Throughput of the reference's own sequential search run for many games at once through one batching evaluator
(sc_game_selfplay_many), against one game through sc_game_selfplay.

BASELINE configs[0] settings (`--rollout-num 20 --num-steps 150 --cpuct 2.5`, noise off, temperature 0) on the
19-block seed-0 network in bf16.  Per run: plies/s, leaf evals/s, mean leaves per device pass and the share of the
game threads' time spent waiting for results.  Writes profiles/evaluator_throughput.json (or --out).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "smart-chess-rust_b200"))


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in q.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as ex:  # noqa: BLE001 - recorded, not fatal
        return {"gpu": "unknown", "power_limit": "unknown", "error": str(ex)}


def main():
    import scb200

    ap = argparse.ArgumentParser()
    ap.add_argument("--games", default="1,15,64,256,2048")
    ap.add_argument("--num-steps", type=int, default=150)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "evaluator_throughput.json"))
    a = ap.parse_args()
    games = [int(x) for x in a.games.split(",")]
    res = {"workload": "configs[0]: rollout_num 20, cpuct 2.5, noise off, temperature 0, num_steps %d; 19-block seed-0 "
                       "net, bf16" % a.num_steps, **gpu_info(), "runs": []}
    kw = dict(rollout_num=20, num_steps=a.num_steps, cpuct=2.5)
    with tempfile.TemporaryDirectory() as d:
        blob = os.path.join(d, "seed0.scw")
        scb200.write_blob(scb200.random_init_state_dict(19, 0), blob)
        eng = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, max(games))
        scb200.game_selfplay(eng, num_steps=4, **{k: v for k, v in kw.items() if k != "num_steps"})  # warm-up
        t0 = time.perf_counter()
        tr = scb200.game_selfplay(eng, seed=0, **kw)
        dt = time.perf_counter() - t0
        plies = len(tr["steps"])
        # (sc_game_selfplay counts no leaf evaluations; the 1-game evaluator run below gives that rate)
        base = {"mode": "sc_game_selfplay", "games": 1, "seconds": dt, "plies": plies, "plies_per_s": plies / dt}
        print(json.dumps(base), flush=True)
        res["baseline"] = base
        for n in games:
            # noise off and temperature 0: the seed changes nothing, every game is the configs[0] game
            seeds = list(range(n))
            t0 = time.perf_counter()
            traces, c = scb200.game_selfplay_many(eng, seeds, **kw)
            dt = time.perf_counter() - t0
            plies = sum(len(t["steps"]) for t in traces)
            r = {"mode": "sc_game_selfplay_many", "games": n, "seconds": dt, "plies": plies, "plies_per_s": plies / dt,
                 "leaf_evals": c["leaves"], "leaf_evals_per_s": c["leaves"] / dt, "passes": c["passes"],
                 "mean_batch": c["leaves"] / max(1, c["passes"]), "largest_batch": c["largest_batch"],
                 "wait_share": c["wait_seconds"] / (n * dt), "speedup_plies_per_s": (plies / dt) / base["plies_per_s"]}
            print(json.dumps(r), flush=True)
            res["runs"].append(r)
        eng.close()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
