"""`scripts/leader-board` + `scripts/show-result` + `scripts/elo.py` for the B200 backend: two networks play N
games with each colour assignment (W as White, then the players swapped), traces go to `${PREFIX}/w_{k}.json`
and `${PREFIX}/b_{k}.json`, each half ends with show-result's `total / white / black` line, and the Elo
difference of the first network is printed as elo.py does.  Defaults are the script's (ROLLOUT 100,
TEMPERATURE 0, TEMPERATURE_SWITCH 0, CPUCT 1.5, 100 games per half).

    python -m scb200.leader_board -W new.scw -B old.scw --temperature-switch 8

Orchestration only: the games are played by the native arena driver (csrc/host/search.cpp)."""
from __future__ import annotations

import argparse
import json
import os


def play_half(white, black, n_games, prefix, tag, a):
    from . import Arena

    ar = Arena(white, black, n_trees=max(1, min(a.trees, n_games)), rollout=a.rollout, cpuct=a.cpuct,
               temperature=a.temperature, temperature_switch=a.temperature_switch, max_plies=a.max_plies,
               seed=a.seed * 2 + (1 if tag == "b" else 0),   # the colour-swapped half draws from its own RNG streams
               n_threads=a.threads or (os.cpu_count() or 8), keep_traces=True,
               pipeline_groups=2 if min(a.trees, n_games) >= 2 else 1)
    st = ar.run(max_games=n_games)
    for k in range(n_games):
        tr = ar.trace(k)
        if tr is None:
            break
        with open(os.path.join(prefix, f"{tag}_{k + 1}.json"), "w") as f:
            json.dump(tr, f)
        if tr["outcome"] is not None:
            print(f"{prefix}/{tag}_{k + 1}.json, {json.dumps(tr['outcome'], separators=(',', ':'))}, num-steps: {len(tr['steps'])}")
    ar.close()
    total, w, b = st["games_finished"], st["white_wins"], st["black_wins"]
    print(f"{total} / {w} / {b}")
    return total, w, b


def main(argv=None):
    from . import Engine, SC_MODE_BF16, SC_MODE_FP16, SC_MODE_FP8, elo

    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("-W", "--white-checkpoint", required=True)
    ap.add_argument("-B", "--black-checkpoint", required=True)
    ap.add_argument("-N", "--games", type=int, default=100, help="games per colour assignment")
    ap.add_argument("--prefix", default=os.environ.get("PREFIX", "replay"))
    ap.add_argument("--rollout", type=int, default=int(os.environ.get("ROLLOUT", 100)))
    ap.add_argument("--temperature", type=float, default=float(os.environ.get("TEMPERATURE", 0)))
    ap.add_argument("--temperature-switch", type=int, default=int(os.environ.get("TEMPERATURE_SWITCH", 0)))
    ap.add_argument("--cpuct", type=float, default=float(os.environ.get("CPUCT", 1.5)))
    ap.add_argument("--max-plies", type=int, default=200)
    ap.add_argument("--trees", type=int, default=2048)
    ap.add_argument("--threads", type=int, default=0)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--device", type=int, default=0)
    prec = ap.add_mutually_exclusive_group()
    prec.add_argument("--fp16", action="store_true", help="fp16 tensor-core operands instead of bf16 for both engines")
    prec.add_argument("--fp8", action="store_true", help="fp8 (e4m3) tensor-core operands instead of bf16 for both engines")
    a = ap.parse_args(argv)

    # under torchrun every rank plays its share of the games on its own GPU (games are independent: no collective
    # until the final tally)
    from .shard import games_for_rank, rank_seed

    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    if world > 1:
        a.device = int(os.environ.get("LOCAL_RANK", 0))
        a.seed = rank_seed(a.seed, rank)
        a.prefix = os.path.join(a.prefix, f"rank{rank}")
        a.threads = a.threads or max(1, (os.cpu_count() or 8) // world)
    n_games = games_for_rank(a.games, rank, world)
    os.makedirs(a.prefix, exist_ok=True)
    tallies = [0] * 6
    if n_games > 0:
        mb = max(1, min(a.trees, n_games))
        mode = SC_MODE_FP16 if a.fp16 else SC_MODE_FP8 if a.fp8 else SC_MODE_BF16
        ea = Engine(a.white_checkpoint, a.device, mode, mb)
        eb = Engine(a.black_checkpoint, a.device, mode, mb)
        print(f"Results are saved in {a.prefix}")
        t1, w1, b1 = play_half(ea, eb, n_games, a.prefix, "w", a)
        print("Swapping the players")
        t2, w2, b2 = play_half(eb, ea, n_games, a.prefix, "b", a)
        ea.close()
        eb.close()
        tallies = [t1, w1, b1, t2, w2, b2]
    if world > 1:
        import torch
        import torch.distributed as dist

        dist.init_process_group("gloo")
        t = torch.tensor(tallies, dtype=torch.int64)
        dist.all_reduce(t)
        tallies = [int(x) for x in t]
        dist.destroy_process_group()
        if rank != 0:
            return 0
    t1, w1, b1, t2, w2, b2 = tallies
    total, win, lost = t1 + t2, w1 + b2, b1 + w2            # from the first network's point of view
    print(f"{a.white_checkpoint}: {total}/{win}/{lost}")
    if 0 < win + (total - win - lost) / 2 < total:
        print(f"ELO: {elo(total, win, lost):+0.2f}")
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
