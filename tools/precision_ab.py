"""bf16 against fp16 (or any list of --modes) tensor-core mode on the bench.py workload (19 blocks, seed-0 net,
seeded random-play leaves).

Alternates engines of the --modes (default bf16,fp16) for --rounds rounds each and measures, per round:
  * the device-resident 2048-leaf step (sc_eval_device), CUDA events per step, L2 flushed between timed steps as
    bench.py does, with nvidia-smi SM clock samples during that leg;
  * sc_eval latency (host buffers) at n = 1 / 8 / 64.
Then both modes' max |d prior| / |d value| against an fp32 engine on the same batch.  Records the card name and power
limit, prints one JSON line and writes it under profiles/ (--out).

--detail adds, per round, the whole-tower launch time from CUDA events (level-2 timing, after the timed window) and
the TFLOP/s it achieves; and per mode, against the fp32 engine, the mean prior error, the mean per-leaf total-variation
distance of the priors, the value error and the rate at which the highest-prior move is the fp32 engine's; and for an
fp8 engine the share of activation elements saturated at +-448 in each layer's output (sc_debug_tower, 256 leaves).

    python tools/precision_ab.py --out profiles/fp16_ab.json
    python tools/precision_ab.py --modes bf16,fp8 --detail --rounds 3 --out profiles/fp8_precision_ab.json
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
import torch  # noqa: E402

import scb200  # noqa: E402
from bench import ClockSampler, make_blob, make_workload  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


MODES = {"bf16": scb200.SC_MODE_BF16, "fp16": scb200.SC_MODE_FP16, "fp8": scb200.SC_MODE_FP8}
# data-sheet dense tensor-core rates of one B200 (1000 W), TFLOP/s
DATASHEET_TFLOPS = {"bf16": 2250.0, "fp16": 2250.0, "fp8": 4500.0}


def leg(blob, mode, pos, moves, off, steps, warmup, detail=False):
    B, n_moves = len(pos), int(off[-1])
    eng = scb200.Engine(blob, 0, mode, B)
    dev = "cuda:0"
    stream = torch.cuda.Stream()
    d_pos = torch.from_numpy(pos.view(np.uint8)).to(dev)
    d_moves = torch.from_numpy(moves.view(np.uint8)).to(dev)
    d_off = torch.from_numpy(off).to(dev)
    d_pri = torch.zeros(n_moves, dtype=torch.float32, device=dev)
    d_val = torch.zeros(B, dtype=torch.float32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {}
    try:
        for nb in (1, 8, 64):
            for it in range(10 + 100):
                if it == 10:
                    t0 = time.perf_counter()
                eng.eval(pos[:nb], moves[: off[nb]], off[: nb + 1])
            out["eval_n%d_us" % nb] = (time.perf_counter() - t0) / 100 * 1e6
        with torch.cuda.stream(stream):
            for _ in range(warmup):
                eng.eval_device(B, d_pos, d_moves, d_off, n_moves, d_pri, d_val, stream.cuda_stream)
            stream.synchronize()
            sampler = ClockSampler(0)
            sampler.start()
            ms = []
            for _ in range(steps):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                eng.eval_device(B, d_pos, d_moves, d_off, n_moves, d_pri, d_val, stream.cuda_stream)
                e1.record(stream)
                e1.synchronize()
                ms.append(e0.elapsed_time(e1))
            clocks = sampler.stop()
        out["step_ms_median"] = statistics.median(ms)
        out["leaves_per_s"] = B / (out["step_ms_median"] * 1e-3)
        out["sm_mhz_median"] = clocks.get("sm_mhz")
        out["clock_reasons"] = clocks.get("reasons")
        if detail:
            # the whole-tower kernel alone: level-2 timing puts an event pair around its launch
            eng.set_timing(2)
            tms = []
            for _ in range(10):
                flush.zero_()
                eng.eval(pos, moves, off)
                tms.append(eng.kernel_timing()[0])
            eng.set_timing(0)
            out["tower_launch_ms_median"] = statistics.median(tms)
            out["tower_tflops"] = eng.timed_flops_per_leaf() * B / (out["tower_launch_ms_median"] * 1e-3) / 1e12
        pri, val = eng.eval(pos, moves, off)
        return out, pri.copy(), val.copy()
    finally:
        eng.close()


def detail_errors(p, v, p32, v32, off):
    """mean prior error, mean per-leaf total-variation distance (scripts/validate_*.py's metric), value error, and the
    rate at which the highest-prior move is the fp32 engine's"""
    d = np.abs(p - p32)
    tv, top = [], []
    for i in range(len(off) - 1):
        a, b = off[i], off[i + 1]
        if b > a:
            tv.append(0.5 * float(d[a:b].sum()))
            top.append(int(np.argmax(p[a:b]) == np.argmax(p32[a:b])))
    return {"mean_abs_d_prior": float(d.mean()), "mean_tv_distance": float(np.mean(tv)),
            "mean_abs_d_value": float(np.abs(v - v32).mean()), "top_move_agreement": float(np.mean(top))}


def saturation(blob, pos, n_blocks=19):
    """fp8 engine: per tower layer, the share of its output elements at +-448 (e4m3 satfinite).  Layer k of the
    1 + 2 n_blocks + 2 writes x (stem, conv2), t (conv1, policy 1x1) or y (value 1x1)"""
    eng = scb200.Engine(blob, 0, scb200.SC_MODE_FP8, len(pos))
    writes = [0] + [1, 0] * n_blocks + [1, 2]
    try:
        out = []
        for k, w in enumerate(writes, start=1):
            buf = eng.debug_tower(pos, k, 0)[w]
            out.append(float(((buf & 0x7FFF) == 0x5F00).mean()))  # fp16 bits of 448
        return out
    finally:
        eng.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--leaves", type=int, default=2048)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "fp16_precision_ab.json"))
    ap.add_argument("--modes", default="bf16,fp16", help="comma-separated tensor-core modes (bf16, fp16, fp8)")
    ap.add_argument("--detail", action="store_true", help="tower launch times, accuracy metrics, fp8 saturation")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("precision_ab.py needs a CUDA device")
    tmp = tempfile.mkdtemp()
    _, blob = make_blob(tmp)
    pos, moves, off = make_workload(a.leaves, seed=0)
    modes = {k: MODES[k] for k in a.modes.split(",")}
    runs = {k: [] for k in modes}
    outs = {}
    for _ in range(a.rounds):
        for name, mode in modes.items():
            r, pri, val = leg(blob, mode, pos, moves, off, a.steps, a.warmup, a.detail)
            runs[name].append(r)
            outs[name] = (pri, val)
    e = scb200.Engine(blob, 0, scb200.SC_MODE_FP32, a.leaves)
    try:
        p32, v32 = e.eval(pos, moves, off)
    finally:
        e.close()
    err = {name: {"max_abs_d_prior": float(np.abs(p - p32).max()), "max_abs_d_value": float(np.abs(v - v32).max())}
           for name, (p, v) in outs.items()}
    if a.detail:
        for name, (p, v) in outs.items():
            err[name].update(detail_errors(p, v, p32, v32, off))
            for r in runs[name]:
                if "tower_tflops" in r:
                    r["tower_tflops_of_datasheet_%s" % name] = r["tower_tflops"] / DATASHEET_TFLOPS[name]
                    r["tower_tflops_of_datasheet_bf16"] = r["tower_tflops"] / DATASHEET_TFLOPS["bf16"]
            if name == "fp8":
                err[name]["saturated_share_per_layer"] = saturation(blob, pos[:256])
    res = {"what": "%s tensor-core mode, 19 blocks, %d leaves, alternating engines" % (" vs ".join(modes), a.leaves),
           "card": card(), "rounds": runs, "error_vs_fp32_engine": err}
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
