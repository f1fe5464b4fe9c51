"""`scripts/run_batch` for the B200 backend: N self-play games on one GPU (or one shard of them per rank
under torchrun), traces written as `${PREFIX}/trace{k}.json` in the format of src/trace.rs:23-32, then the
per-game summary lines the reference script prints.  Flags are the `selfplay` binary's (src/main.rs:25-60)
plus --trees (concurrent games per GPU) and -N (games).

    python -m scb200.run_batch -c model.scw -N 500 --rollout-num 180 --temperature-switch 4 --cpuct 2.5

This is orchestration only: the games are played by the native driver (csrc/host/search.cpp)."""
from __future__ import annotations

import argparse
import json
import os


def main(argv=None):
    from . import Engine, SelfPlay, SC_MODE_BF16, SC_MODE_FP16, SC_MODE_FP32, SC_MODE_FP8
    from .shard import game_ids_for_rank, rank_seed

    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("-c", "--checkpoint", required=True, help=".scw weight blob (python -m scb200.export)")
    ap.add_argument("-N", "--games", type=int, default=int(os.environ.get("N", 100)))
    ap.add_argument("--prefix", default=os.environ.get("PREFIX", "."))
    ap.add_argument("--trees", type=int, default=2048)
    ap.add_argument("--rollout-num", type=int, default=300)
    ap.add_argument("-n", "--num-steps", type=int, default=100)
    ap.add_argument("--temperature", type=float, default=0.0)
    ap.add_argument("--cpuct", type=float, default=1.0)
    ap.add_argument("--temperature-switch", type=int, default=30)
    ap.add_argument("--epsilon", type=float, default=0.15)
    prec = ap.add_mutually_exclusive_group()
    prec.add_argument("--fp32", action="store_true", help="parity mode (FP32 FFMA) instead of bf16 tensor cores")
    prec.add_argument("--fp16", action="store_true",
                      help="fp16 tensor-core operands instead of bf16 (the precision of a 16-mixed trained net)")
    prec.add_argument("--fp8", action="store_true",
                      help="fp8 (e4m3) tensor-core operands instead of bf16 (throughput mode, lower precision)")
    ap.add_argument("--leaves-per-tree", type=int, default=1,
                    help="1 = the reference's sequential search; K > 1 = K leaves per tree per batch (virtual loss); "
                         "-1 = 1 until games run out, then the remaining games share the batch")
    ap.add_argument("--threads", type=int, default=0)
    ap.add_argument("--seed", type=int, default=0)
    a = ap.parse_args(argv)

    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    mine = game_ids_for_rank(a.games, rank, world)        # game ids of this shard (game g -> rank g mod world)
    if len(mine) == 0:
        return 0
    trees = max(1, min(a.trees, len(mine)))
    kl = max(1, a.leaves_per_tree)
    mode = SC_MODE_FP32 if a.fp32 else SC_MODE_FP16 if a.fp16 else SC_MODE_FP8 if a.fp8 else SC_MODE_BF16
    eng = Engine(a.checkpoint, local, mode, trees * kl)
    sp = SelfPlay(eng, n_trees=trees, rollout_num=a.rollout_num, num_steps=a.num_steps, cpuct=a.cpuct, epsilon=a.epsilon,
                  with_noise=True, temperature_switch=a.temperature_switch, temperature=a.temperature,
                  seed=rank_seed(a.seed, rank), n_threads=a.threads or max(1, (os.cpu_count() or 8) // world),
                  pipeline_groups=2 if trees >= 2 else 1, keep_traces=True, leaves_per_tree=a.leaves_per_tree)
    st = sp.run(max_games=len(mine))
    os.makedirs(a.prefix, exist_ok=True)
    for k in range(len(mine)):
        tr = sp.trace(k)
        if tr is None:
            break
        gid = mine[sp.trace_game(k)]          # the file is named after the GAME (its id in the run), not its finishing order
        with open(os.path.join(a.prefix, f"trace{gid + 1}.json"), "w") as f:
            json.dump(tr, f)
        print(f"{gid + 1:02d}, {json.dumps(tr['outcome'], separators=(',', ':'))}, num-steps: {len(tr['steps'])}")
    print(f"# rank {rank}: {st['games_finished']} games, {st['moves']} plies, {st['leaf_evals'] / max(st['seconds'], 1e-9):.0f} "
          f"leaf evals/s, W/B/D {st['white_wins']}/{st['black_wins']}/{st['draws']}")
    sp.close()
    eng.close()
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
