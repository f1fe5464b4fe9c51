#!/usr/bin/env python
"""bench.py -- leaf evals/s of the B200 leaf-evaluation backend (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm
    python bench.py --impl reference --gpus N --steps K ...   # CPU reference arm (oracle port)

A "step" is one pass of the hot path over one batch: B leaves (one per concurrent search tree,
BASELINE.json configs[2]: 2048 concurrent trees on 1xB200) -> plane encode -> 19-block
policy/value network -> move-index gather + renormalisation -> priors/values.  Positions are
seeded random play with true 8-ply history; the network is the seed-0 random init of the
reference's architecture (no checkpoints offline).  N > 1: leaves (games) are sharded across
ranks, no data-path collective ("scaling": "weak").

value   = leaves/s with inputs already resident in HBM (sc_eval_device), CUDA events per step,
          L2 flushed between timed steps, max over ranks.
e2e     = same metric through the C-ABI call a Rust shim makes (sc_eval) with pinned HOST
          buffers: H2D of positions/moves and D2H of priors/values inside the timed region.
roofline= the dominant kernel (3x3 256->256 tcgen05 conv): algorithmic FLOPs per launch /
          its average launch duration measured with CUDA event pairs during the timed steps.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "smart-chess-rust_b200"))

FLOP_PER_LEAF = 2 * 1463895040            # BASELINE.md section 2
FLOP_PER_LEAF_CONV3 = 2 * 64 * 256 * 2304  # one 3x3 256->256 layer, per leaf
N_BLOCKS = 19
DUMP_BYTES = 64_000_000                    # --dump-outputs: at most this much over all ranks, headers included
NPY_HEADER = 128                           # bytes before the data of a 1-D .npy file


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"tflops": d.get("bf16_tflops_sustained", 1371.0), "tflops_burst": d.get("bf16_tflops", 1666.7),
                "hbm_gbs": d.get("hbm_gbs", 6547.8), "src": "measured",
                "sustained_sm_mhz": (d.get("clocks_under_load") or {}).get("sm_mhz_median")}
    return {"tflops": 1400.0, "tflops_burst": 1590.0, "hbm_gbs": 6650.0, "src": "fallback", "sustained_sm_mhz": 1300.0}


# ------------------------------------------------------------------------------------------
# synthetic workload of OUR arm: positions from the driver's native rules (sc_random_positions), weights
# from scb200.random_init -- nothing under oracle/ is imported on this arm.  The cpu_baseline leg and the
# --impl reference arm draw their own bounded sample of the same workload from the oracle.
# ------------------------------------------------------------------------------------------
def make_workload(n_leaves: int, seed: int):
    import scb200

    pos, moves, off = scb200.random_positions(n_leaves, seed=seed, max_ply=150)
    return pos, moves, off


def make_blob(tmpdir: str, n_blocks: int = N_BLOCKS):
    import scb200

    sd = scb200.random_init_state_dict(n_blocks, 0)   # == load_model(n_res_blocks=19) seed-0 init (py/module.py:184-212)
    path = os.path.join(tmpdir, f"seed0_{n_blocks}.scw")
    scb200.write_blob(sd, path)
    return sd, path


def dump_outputs(out_dir: str, pri, val, off, rank: int, world: int):
    """Writes what one step returns to its caller: priors.npy (float32, per legal move, leaf after leaf) and values.npy
    (float32, per leaf), with leaves.npy (each leaf's index in the step) and offsets.npy (where each leaf's priors start
    in priors.npy, plus the end), both float64.  Above DUMP_BYTES, a fixed seeded sample of whole leaves in leaf order."""
    import numpy as np

    names = ("priors", "values", "leaves", "offsets")
    budget = DUMP_BYTES // world - len(names) * NPY_HEADER - 8   # bytes per rank, less the headers and the end offset
    lens = np.diff(off).astype(np.int64)
    leaves = np.arange(len(val))
    if 4 * int(lens.sum()) + 20 * len(val) > budget:
        order = np.random.default_rng(0).permutation(len(val))
        cost = np.cumsum(4 * lens[order] + 20)      # a leaf's priors and value (float32), index and offset (float64)
        leaves = np.sort(order[: int(np.searchsorted(cost, budget, side="right"))])
    lens = lens[leaves]
    starts = np.concatenate([[0], np.cumsum(lens)])
    pri = pri[np.arange(int(starts[-1])) + np.repeat(off[leaves] - starts[:-1], lens)]
    arrays = (pri.astype(np.float32), val[leaves].astype(np.float32), leaves.astype(np.float64), starts.astype(np.float64))
    os.makedirs(out_dir, exist_ok=True)
    suffix = "" if world == 1 else f"_rank{rank}"
    for name, a in zip(names, arrays):
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), a)


def oracle_sample(n: int, seed: int):
    """bounded sample of the same workload for the CPU legs (seeded random play with true history)"""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import chess_oracle as co

    return co.random_play_positions(n, seed=seed)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------
# CPU baseline (oracle port of the reference path, timed on the box's host cores)
# ------------------------------------------------------------------------------------------
def cpu_reference_throughput(sd, games, budget_s: float, batch: int):
    """encode (C oracle) + module.py forward restated in torch fp32 on CPU + post_process, on a
    bounded sample of the workload.  Returns (leaves/s batched, leaves/s at batch 1, n, threads)."""
    import numpy as np
    import torch

    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import chess_oracle as co
    import net

    def run(sub):
        planes = np.stack([g.encode()[0] for g in sub])
        meta = np.stack([g.encode()[1] for g in sub])
        lp, v = net.forward(sd, net.planes_i8_hwc_to_nchw(planes), torch.from_numpy(meta).float())
        lp = lp.numpy()
        for i, g in enumerate(sub):
            co.post_process(lp[i], g.move_indices())
        return v

    run(games[:min(batch, 8)])  # warm-up
    done, t0 = 0, time.perf_counter()
    while True:
        sub = [games[(done + i) % len(games)] for i in range(batch)]
        run(sub)
        done += batch
        el = time.perf_counter() - t0
        if el >= budget_s:
            break
    batched = done / el
    # the reference's real operating point: one position per forward (torch.rs:119 unsqueeze(0))
    n1, t1 = 0, time.perf_counter()
    while time.perf_counter() - t1 < min(4.0, budget_s / 3):
        run([games[n1 % len(games)]])
        n1 += 1
    b1 = n1 / (time.perf_counter() - t1)
    return batched, b1, done, torch.get_num_threads()


def cpu_reference_selfplay(sd, budget_s: float):
    """The reference's self-play loop on the CPU (sequential search of src/mcts.rs restated in the oracle, one
    leaf per forward): plies/s at 180 rollouts/move, (i) as the reference runs it -- `select` calls `predict` at
    every level of every descent -- and (ii) with the priors cached on the children."""
    import torch

    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import chess_oracle as co
    import net

    def ev(game, depth, moves):
        planes, meta = game.encode(depth)
        with torch.no_grad():
            lp, v = net.forward(sd, net.planes_i8_hwc_to_nchw(planes[None]), torch.from_numpy(meta[None]).float())
        return co.post_process(lp[0].numpy(), game.move_indices(moves)), float(v[0, 0])

    t = co.Tree(ev)
    t0 = time.perf_counter()
    rollouts = 0
    while time.perf_counter() - t0 < budget_s:
        t.search(10, 2.5)            # 10 more rollouts on the same root
        rollouts += 10
    el = time.perf_counter() - t0
    evals, predicts = t.n_evals, t.n_predicts
    cached = rollouts / el / 180.0
    faithful = cached * evals / max(predicts, 1)
    return {"plies_per_s_priors_cached": cached, "plies_per_s_predict_every_level": faithful,
            "rollouts_timed": rollouts, "network_evals": evals, "predict_calls_of_the_reference": predicts}


def reference_arm(args):
    """`--impl reference`: the reference's CPU implementation of the path.  The Rust binary cannot
    be built here (no cargo; python-chess and tch-rs absent), so this is the oracle port: the
    reference's module.py arithmetic on libtorch CPU + chess.rs/queenmoves.rs semantics in C."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch

    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import net

    torch.set_num_threads(os.cpu_count() or 1)   # torchrun exports OMP_NUM_THREADS=1; use every host core
    sd = net.init_state_dict(N_BLOCKS, 0)
    import numpy as np
    import chess_oracle as co

    chunk = 64                                    # leaves per forward (batched far beyond the reference's batch 1)
    games = oracle_sample(min(args.leaves, 512), seed=1000)
    steps, warm = args.steps, args.warmup

    def forward_chunk(sub):
        planes = np.stack([g.encode()[0] for g in sub])
        meta = np.stack([g.encode()[1] for g in sub])
        lp, v = net.forward(sd, net.planes_i8_hwc_to_nchw(planes), torch.from_numpy(meta).float())
        lp = lp.numpy()
        for i, g in enumerate(sub):
            co.post_process(lp[i], g.move_indices())

    for _ in range(max(warm, 1)):                 # warm-up: one chunk each
        forward_chunk(games[:chunk])
    t0 = time.perf_counter()
    forward_chunk(games[:chunk])
    rate = chunk / (time.perf_counter() - t0)
    # a step = the arm's leaves_per_step when K steps of it fit ~150 s of CPU work, else the largest bounded sample that does
    budget = 150.0
    per_step = args.leaves
    if steps * per_step / rate > budget:
        per_step = max(chunk, int(budget * rate / steps) // chunk * chunk)

    def step():
        for lo in range(0, per_step, chunk):
            forward_chunk([games[(lo + i) % len(games)] for i in range(min(chunk, per_step - lo))])

    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    el = time.perf_counter() - t0
    v = steps * per_step / el
    # the reference's real operating point: one position per forward (src/backends/torch.rs:119 unsqueeze(0))
    n1, t1 = 0, time.perf_counter()
    while time.perf_counter() - t1 < 3.0:
        forward_chunk([games[n1 % len(games)]])
        n1 += 1
    b1 = n1 / (time.perf_counter() - t1)
    line = {
        "impl": "reference", "metric": "leaf_evals_per_s", "value": v, "unit": "leaf evals/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": el / steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.leaves),
        "cpu_baseline": {"value": v, "unit": "leaf evals/s", "cores": torch.get_num_threads(), "kind": "port",
                         "leaves_per_step_run": per_step, "batch1_value": b1,
                         "sample": f"{per_step} leaves per step (of the {args.leaves}-leaf step of config), evaluated as "
                                   f"forwards of {chunk} leaves, fp32 libtorch CPU on all host threads; batch1_value = "
                                   f"one leaf per forward, the reference's own operating point"},
        "e2e": {"value": v, "unit": "leaf evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def workload_config(leaves):
    return {"workload": f"batched leaf eval, {leaves} leaves/step = one leaf per concurrent search tree "
                        f"(BASELINE configs[2]: 2048 concurrent trees, 19-block LayerNorm+SE net, "
                        f"seeded random-play positions with 8-ply history)",
            "leaves_per_step": leaves, "n_res_blocks": N_BLOCKS, "l2": "flushed between timed steps (256 MiB memset); the separate sustained leg runs back to back",
            "parallelism": "leaves sharded by game, one process per GPU, no collective on the data path"}


# ------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--leaves", type=int, default=2048, help="leaves per step per GPU")
    ap.add_argument("--mode", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of CPU baseline work (rank 0, N=1)")
    ap.add_argument("--selfplay-moves", type=int, default=16384, help="plies of batched self-play to time (0 = skip)")
    ap.add_argument("--leaves-per-tree", type=int, default=1,
                    help="self-play leg: leaves per tree per batch (1 = the reference's sequential search; "
                         ">1 = virtual loss, leaves/K trees)")
    ap.add_argument("--arena-seconds", type=float, default=0.0,
                    help="also time the leader-board mode (BASELINE configs[4]: two random-init nets, rollout 100, "
                         "temperature-switch 8, both colour assignments) for this many seconds per rank (0 = skip)")
    ap.add_argument("--threads", type=int, default=0, help="host worker threads for self-play (0 = cores / ranks)")
    ap.add_argument("--one-leaf-plies", type=int, default=40,
                    help="plies of one game through the one-leaf interface (BASELINE configs[0] settings) to time (0 = skip)")
    ap.add_argument("--sustain", type=float, default=5.0,
                    help="seconds of back-to-back steps for the sustained roofline leg and the clock samples (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the priors and values of the last timed step as DIR/priors.npy and DIR/values.npy "
                         "(float32), with DIR/leaves.npy and DIR/offsets.npy to split the priors by leaf; at most 64 MB "
                         "(a seeded sample of the leaves beyond that); with several ranks, _rank<r> before .npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs dumps the b200 arm's timed step; the reference arm does not keep its outputs")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    if args.impl == "reference":
        reference_arm(args)
        return

    import numpy as np
    import torch

    import scb200

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this backend has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    B, K, W = args.leaves, args.steps, args.warmup
    mode = scb200.SC_MODE_BF16 if args.mode == "bf16" else scb200.SC_MODE_FP32
    tmp = tempfile.mkdtemp(prefix="scb200_bench_")
    sd, blob = make_blob(tmp)
    from scb200 import shard

    pos, moves, off = make_workload(B, seed=shard.rank_seed(1000, rank))
    n_moves = int(off[B])
    eng = scb200.Engine(blob, local_rank, mode, B)

    stream = torch.cuda.Stream(device=local_rank)
    sh = stream.cuda_stream
    # device-resident inputs / outputs
    d_pos = torch.from_numpy(pos.view(np.uint8)).to(f"cuda:{local_rank}")
    d_moves = torch.from_numpy(moves.view(np.uint8)).to(f"cuda:{local_rank}")
    d_off = torch.from_numpy(off).to(f"cuda:{local_rank}")
    d_pri = torch.zeros(n_moves, dtype=torch.float32, device=f"cuda:{local_rank}")
    d_val = torch.zeros(B, dtype=torch.float32, device=f"cuda:{local_rank}")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{local_rank}")
    # pinned host buffers for the e2e leg
    h_pos = torch.from_numpy(pos.view(np.uint8)).pin_memory()
    h_moves = torch.from_numpy(moves.view(np.uint8)).pin_memory()
    h_off = torch.from_numpy(off).pin_memory()
    h_pri = torch.zeros(n_moves, dtype=torch.float32).pin_memory()
    h_val = torch.zeros(B, dtype=torch.float32).pin_memory()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def dev_step():
        eng.eval_device(B, d_pos, d_moves, d_off, n_moves, d_pri, d_val, sh)

    # ---- small-batch latency of the host-buffer call (what the one-leaf `Game::predict` shim sees, src/backends/torch.rs:115-125)
    #      and BASELINE configs[0] through the one-leaf interface.  Measured BEFORE the throughput legs: a single game does
    #      not run next to a saturated, power-capped GPU, and the SM clock takes seconds to come back after such a leg.
    latency, one_leaf = {}, None
    if rank == 0:
        pos_np = h_pos.numpy().view(scb200.POSITION_DTYPE)
        for nb in (1, 2, 8, 16, 64, 128):
            if nb > B:
                continue
            # the caller's arrays are prepared once (numpy views of the pinned buffers): the loop times the call, not slicing
            p_n = pos_np[:nb]
            m_n = h_moves.numpy().view(scb200.MOVE_DTYPE)[: int(h_off[nb])]
            o_n = h_off.numpy()[: nb + 1]
            pr_n, va_n = h_pri.numpy(), h_val.numpy()
            for it in range(10 + 100):
                if it == 10:
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                eng.eval(p_n, m_n, o_n, pr_n, va_n, sh)
            latency["n%d_ms" % nb] = (time.perf_counter() - t0) / 100 * 1e3
        if args.one_leaf_plies > 0:
            t0 = time.perf_counter()
            tr = scb200.game_selfplay(eng, rollout_num=20, num_steps=args.one_leaf_plies, cpuct=2.5, with_noise=False,
                                      temperature_switch=0, temperature=0.0)
            el = time.perf_counter() - t0
            one_leaf = {"plies_per_s": len(tr["steps"]) / el, "plies": len(tr["steps"]), "seconds": el,
                        "config": "BASELINE configs[0] through the reference's one-leaf interface (sc_game_selfplay: predict at "
                                  "every level of every descent, one sc_eval(n=1) per predict): rollout-num 20, cpuct 2.5, "
                                  "first %d plies, %s" % (args.one_leaf_plies, args.mode)}

    # ---- device-resident leg (value) --------------------------------------------------------
    with torch.cuda.stream(stream):
        for _ in range(W):
            dev_step()
        stream.synchronize()
        eng.set_timing(2)       # event pairs around every 3x3 conv launch, read back after the sync
        sampler = ClockSampler(local_rank)
        sampler.start()
        launches0 = eng.launch_count()
        barrier()
        step_ms, conv_ms, conv_n = [], [], 0
        t_wall0 = time.perf_counter()
        for _ in range(K):
            flush.zero_()       # L2 flush, outside the per-step event pair
            ev0 = torch.cuda.Event(enable_timing=True)
            ev1 = torch.cuda.Event(enable_timing=True)
            ev0.record(stream)
            dev_step()          # with timing on, returns after the step's last event completed
            ev1.record(stream)
            ev1.synchronize()
            step_ms.append(ev0.elapsed_time(ev1))
            a, n = eng.kernel_timing()
            conv_ms.append(a * n)   # device time of all timed tower-convolution launches of this step
            conv_n = n
        barrier()
        t_wall = time.perf_counter() - t_wall0
        launches = eng.launch_count() - launches0
        eng_timed_flops = eng.timed_flops_per_leaf()
        # the sustained leg below overwrites d_pri / d_val: keep the last timed step's results
        dumped = (d_pri.cpu().numpy(), d_val.cpu().numpy()) if args.dump_outputs else None
        # ---- sustained leg: the same step back to back for >= args.sustain seconds, no flush, no idle gap beyond the
        #      engine's own event read-back: what the kernel does under continuous load (power cap); its roofline
        #      fraction is taken against the SUSTAINED peak, the event-bracketed steps above against the BURST peak.
        #      The step's activations (~200 MB of bf16 maps at 2048 leaves) exceed nothing the flush would add: inputs
        #      and weights are L2-resident in steady state, as they are in self-play.
        sus = None
        if args.sustain > 0:
            sus_conv_ms, sus_steps = 0.0, 0
            ev0 = torch.cuda.Event(enable_timing=True)
            ev1 = torch.cuda.Event(enable_timing=True)
            ev0.record(stream)
            t_s0 = time.perf_counter()
            while time.perf_counter() - t_s0 < args.sustain:
                dev_step()
                a, n = eng.kernel_timing()
                sus_conv_ms += a * n
                sus_steps += 1
            ev1.record(stream)
            ev1.synchronize()
            sus = {"seconds": ev0.elapsed_time(ev1) * 1e-3, "steps": sus_steps, "conv_ms_total": sus_conv_ms}
        clocks = sampler.stop()
        eng.set_timing(0)
    total_ms = float(sum(step_ms))

    # ---- end-to-end leg through the host-buffer C-ABI call -------------------------------------
    for _ in range(2):
        eng.eval(h_pos.numpy().view(scb200.POSITION_DTYPE), h_moves, h_off, h_pri, h_val, sh)
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        eng.eval(h_pos.numpy().view(scb200.POSITION_DTYPE), h_moves, h_off, h_pri, h_val, sh)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0

    # ---- batched self-play at 180 rollouts (BASELINE configs[2]: 2048 concurrent trees) ---------------
    sp_stats = None
    if args.selfplay_moves > 0:
        nthr = args.threads or max(1, (os.cpu_count() or 8) // max(world, 1))
        eng_sp = scb200.Engine(blob, local_rank, mode, B)
        kl = max(1, args.leaves_per_tree)
        sp = scb200.SelfPlay(eng_sp, n_trees=max(2, B // kl), leaves_per_tree=kl, rollout_num=180, num_steps=150, cpuct=2.5, epsilon=0.15,
                             with_noise=True, temperature_switch=4, temperature=0.0, seed=shard.rank_seed(100, rank),
                             n_threads=nthr, pipeline_groups=2)
        barrier()
        sp_stats = sp.run(max_moves=args.selfplay_moves)
        sp_stats["threads"] = nthr
        sp_stats["trees"] = max(2, B // kl)
        sp.close()
        eng_sp.close()

    # ---- leader-board mode (BASELINE configs[4]), optional ------------------------------------------
    arena = None
    if args.arena_seconds > 0:
        nthr = args.threads or max(1, (os.cpu_count() or 8) // max(world, 1))
        sd_b = scb200.random_init_state_dict(N_BLOCKS, 1)      # the second net: same shape, seed 1
        blob_b = os.path.join(tmp, "seed1.scw")
        scb200.write_blob(sd_b, blob_b)
        ea = scb200.Engine(blob, local_rank, mode, B)
        eb = scb200.Engine(blob_b, local_rank, mode, B)
        tot = {"leaf_evals": 0, "moves": 0, "seconds": 0.0, "games_finished": 0}
        for white, black in ((ea, eb), (eb, ea)):               # both colour assignments (scripts/leader-board:49-54)
            ar = scb200.Arena(white, black, n_trees=B, rollout=100, cpuct=1.5, temperature=0.0, temperature_switch=8,
                              max_plies=200, seed=shard.rank_seed(200, rank), n_threads=nthr, pipeline_groups=2)
            barrier()
            st = ar.run(max_seconds=args.arena_seconds / 2)
            ar.close()
            for k in tot:
                tot[k] += st[k]
        ea.close()
        eb.close()
        t3 = torch.tensor([tot["leaf_evals"], tot["moves"], tot["seconds"]], dtype=torch.float64, device=f"cuda:{local_rank}")
        if dist is not None:
            tmax = t3.clone()
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            dist.all_reduce(t3, op=dist.ReduceOp.SUM)
            t3[2] = tmax[2]
        arena = {"leaf_evals_per_s": float(t3[0] / t3[2]), "plies_per_s": float(t3[1] / t3[2]), "seconds": float(t3[2]),
                 "config": "two random-init 19-block nets (seeds 0 and 1), %d concurrent games per GPU, rollout 100, cpuct 1.5, "
                           "temperature-switch 8, noise off, both colour assignments, host threads = %d per GPU" % (B, nthr)}

    # ---- max over ranks ------------------------------------------------------------------------
    sp_secs = sp_stats["seconds"] if sp_stats else 0.0
    sp_moves = float(sp_stats["moves"]) if sp_stats else 0.0
    sp_evals = float(sp_stats["leaf_evals"]) if sp_stats else 0.0
    if dist is not None:
        t = torch.tensor([total_ms, e2e_s, sp_secs], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_s, sp_secs = float(t[0]), float(t[1]), float(t[2])
        t2 = torch.tensor([sp_moves, sp_evals], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(t2, op=dist.ReduceOp.SUM)
        sp_moves, sp_evals = float(t2[0]), float(t2[1])
    value = world * B * K / (total_ms * 1e-3)
    e2e = world * B * K / e2e_s

    # sanity: the timed output is a real evaluation (not part of the timed region)
    pri_chk = d_pri.cpu().numpy()
    assert np.isfinite(pri_chk).all() and abs(float(pri_chk[: int(off[1])].sum()) - 1.0) < 0.05
    if dumped is not None:
        dump_outputs(args.dump_outputs, *dumped, off, rank, world)

    if rank == 0:
        peaks = _peaks()
        conv_tot_ms = float(np.mean(conv_ms)) if conv_ms else None
        conv_avg_ms = conv_tot_ms / conv_n if conv_tot_ms and conv_n else None
        timed_flops = eng_timed_flops
        roof = None
        if conv_avg_ms and conv_avg_ms > 0:
            ach = B * timed_flops / (conv_tot_ms * 1e-3) / 1e12
            tower = conv_n == 1
            roof = {"bound": "tensor",
                    "kernel": ("tc_gemm_kernel<256, pair, TOWER>: stem + 19 x (conv3x3+LN+ReLU, conv3x3+LN+SE+residual+ReLU) + 2 head 1x1 convs in one launch"
                               if tower else
                               "tc_gemm_kernel<256, EPI_LN | EPI_LN_SE, pair> (3x3 256->256 conv, bias+LN[+SE+residual] fused)"),
                    "achieved": ach, "peak": peaks["tflops_burst"], "unit": "TFLOP/s", "frac": ach / peaks["tflops_burst"],
                    "peak_kind": f"bf16_tflops burst ({peaks['src']}): each timed step is bracketed by CUDA events and preceded by "
                                 f"an L2 flush + sync, i.e. the kernel is timed alone",
                    # not measured by this run: dram__bytes_read.sum + dram__bytes_write.sum of one launch from the committed
                    # ncu --set full capture of this workload
                    "traffic": (0.750e9 if tower else (95.4e6 + 161.0e6) / 2) if B == 2048 and args.mode == "bf16" else None,
                    "traffic_source": "constant: ncu --set full capture profiles/r02_tower_full_raw.csv (236 MB read + 514 MB "
                                      "written per whole-tower launch; 1644 MB in round 1, profiles/r02_tile_groups.md); not "
                                      "re-measured by this run",
                    "launches_timed_per_step": conv_n, "avg_launch_ms": conv_avg_ms,
                    "flops_per_launch": B * timed_flops / conv_n,
                    "whole_step_tflops": value / world * FLOP_PER_LEAF / 1e12}
            if sus and sus["conv_ms_total"] > 0:
                ach_s = sus["steps"] * B * timed_flops / (sus["conv_ms_total"] * 1e-3) / 1e12
                roof["sustained"] = {
                    "achieved": ach_s, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": ach_s / peaks["tflops"],
                    "peak_kind": f"bf16_tflops_sustained ({peaks['src']}): {sus['steps']} steps back to back over "
                                 f"{sus['seconds']:.1f} s, no flush, kernel time from the same event pairs",
                    "leaf_evals_per_s": sus["steps"] * B / sus["seconds"], "seconds": sus["seconds"], "steps": sus["steps"],
                    "avg_launch_ms": sus["conv_ms_total"] / sus["steps"] / conv_n}
                # the sustained peak is a cuBLAS loop under the 1 kW cap; MEASURED_PEAKS.json records the SM clock it settled
                # at.  A kernel that spends less energy per FLOP is capped at a higher clock, so its fraction of that peak can
                # exceed 1; the same fraction at equal clocks is printed beside it.
                if peaks.get("sustained_sm_mhz") and clocks.get("sm_mhz"):
                    roof["sustained"]["peak_measured_at_sm_mhz"] = peaks["sustained_sm_mhz"]
                    roof["sustained"]["this_run_sm_mhz"] = clocks["sm_mhz"]
                    roof["sustained"]["frac_at_equal_clock"] = roof["sustained"]["frac"] * peaks["sustained_sm_mhz"] / clocks["sm_mhz"]
            if args.mode == "fp32":
                # BASELINE.md section 2: the fp32 peaks are not in MEASURED_PEAKS.json -- measure them on this box, the way the
                # driver measured the bf16 one (torch.matmul 8192^3, best of 5, CUDA events): FP32 on the CUDA cores (cuBLAS
                # SGEMM, TF32 off) and TF32 on the tensor cores
                def _matmul_peak(tf32):
                    old = torch.backends.cuda.matmul.allow_tf32
                    torch.backends.cuda.matmul.allow_tf32 = tf32
                    a = torch.randn(8192, 8192, device=f"cuda:{local_rank}")
                    b = torch.randn(8192, 8192, device=f"cuda:{local_rank}")
                    best = 0.0
                    for it in range(6):
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        torch.matmul(a, b)
                        e1.record()
                        e1.synchronize()
                        if it:
                            best = max(best, 2 * 8192 ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
                    torch.backends.cuda.matmul.allow_tf32 = old
                    return best
                ffma_peak, tf32_peak = _matmul_peak(False), _matmul_peak(True)
                roof["fp32_peaks_measured_here"] = {
                    "fp32_ffma_tflops": ffma_peak, "tf32_tflops": tf32_peak, "how": "torch.matmul fp32 8192^3, best of 5, TF32 off / on",
                    "achieved_over_fp32_ffma_peak": ach / ffma_peak if ffma_peak else None,
                    "achieved_over_tf32_peak_div_3": ach / (tf32_peak / 3) if tf32_peak else None}
                roof["kernel"] = ("tc_gemm_kernel<256, EPI_F32, pair>: 3x3 256->256 conv as a bf16x3 split GEMM (6 tcgen05 bf16 products "
                                  "per fp32 product, fp32 accumulate in TMEM), one launch per layer; LayerNorm / SE in fp32 kernels")
                roof["traffic"] = None
                # FP32 parity mode: the same kernel runs the bf16x3 operand split (6 tensor-core products per fp32
                # product), so its ceiling is the bf16 peak / 6; achieved counts fp32 FLOPs
                roof["peak"] = peaks["tflops_burst"] / 6
                roof["frac"] = ach / roof["peak"]
                roof["peak_kind"] = (f"bf16_tflops burst ({peaks['src']}) / 6: fp32 products as 6 bf16 tensor-core products "
                                     f"(3-way operand split, terms below 2^-16 dropped)")
                if "sustained" in roof:
                    roof["sustained"]["peak"] = peaks["tflops"] / 6
                    roof["sustained"]["frac"] = roof["sustained"]["achieved"] / roof["sustained"]["peak"]
                    if "frac_at_equal_clock" in roof["sustained"]:
                        roof["sustained"]["frac_at_equal_clock"] = (roof["sustained"]["frac"] * roof["sustained"]["peak_measured_at_sm_mhz"]
                                                                    / roof["sustained"]["this_run_sm_mhz"])
        cpu = None
        if world == 1 and args.cpu_budget > 0:
            b, b1, n, thr = cpu_reference_throughput(sd, oracle_sample(512, seed=1000), args.cpu_budget, 64)
            cpu = {"value": b, "unit": "leaf evals/s", "cores": thr, "kind": "port",
                   "sample": f"{n} leaves of the same workload in batches of 64 (fp32 libtorch CPU oracle)",
                   "batch1_value": b1, "host_cpus": os.cpu_count(),
                   "selfplay_180_rollouts": cpu_reference_selfplay(sd, min(5.0, args.cpu_budget / 2))}
        h2d = int(pos.nbytes + moves.nbytes + off.nbytes)
        d2h = int(n_moves * 4 + B * 4)
        line = {
            "metric": "leaf_evals_per_s", "value": value, "unit": "leaf evals/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": args.mode, "data": "synthetic", "config": workload_config(B),
            "e2e": {"value": e2e, "unit": "leaf evals/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
            "wall_s_timed_region": t_wall, "call_latency": latency, "one_leaf_game": one_leaf,
        }
        if sp_stats:
            line["selfplay"] = {
                "moves_per_s": sp_moves / sp_secs, "leaf_evals_per_s": sp_evals / sp_secs, "unit": "plies/s at 180 rollouts/move",
                "config": "%d concurrent trees per GPU x %d leaves per tree per batch%s, rollout-num 180, cpuct 2.5, "
                          "temperature-switch 4, epsilon 0.15 noise on, two pipeline groups, host threads = %d per GPU"
                          % (sp_stats["trees"], max(1, args.leaves_per_tree),
                             "" if args.leaves_per_tree <= 1 else " (virtual loss; not the reference's visit counts)",
                             sp_stats["threads"]),
                "plies": sp_moves, "seconds": sp_secs, "device_wait_frac_rank0": sp_stats["wait_seconds"] / sp_stats["seconds"],
                "roofline": {"bound": "tensor", "achieved": sp_evals / sp_secs / world * FLOP_PER_LEAF / 1e12,
                             "peak": peaks["tflops"], "unit": "TFLOP/s",
                             "frac": sp_evals / sp_secs / world * FLOP_PER_LEAF / 1e12 / peaks["tflops"],
                             "peak_kind": "bf16_tflops_sustained: whole path (search on the host + every kernel), per GPU"},
                "games_finished_rank0": sp_stats["games_finished"],
            }
        if arena:
            line["arena"] = arena
        print(json.dumps(line), flush=True)
    eng.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
