"""bf16 against fp16 tensor-core mode on the bench.py workload (19 blocks, seed-0 net, seeded random-play leaves).

Alternates a bf16 and an fp16 engine for --rounds rounds each and measures, per round:
  * the device-resident 2048-leaf step (sc_eval_device), CUDA events per step, L2 flushed between timed steps as
    bench.py does, with nvidia-smi SM clock samples during that leg;
  * sc_eval latency (host buffers) at n = 1 / 8 / 64.
Then both modes' max |d prior| / |d value| against an fp32 engine on the same batch.  Records the card name and power
limit, prints one JSON line and writes it under profiles/ (--out).

    python tools/precision_ab.py --out profiles/fp16_ab.json
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


def leg(blob, mode, pos, moves, off, steps, warmup):
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
        pri, val = eng.eval(pos, moves, off)
        return out, pri.copy(), val.copy()
    finally:
        eng.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--leaves", type=int, default=2048)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "fp16_precision_ab.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("precision_ab.py needs a CUDA device")
    tmp = tempfile.mkdtemp()
    _, blob = make_blob(tmp)
    pos, moves, off = make_workload(a.leaves, seed=0)
    modes = {"bf16": scb200.SC_MODE_BF16, "fp16": scb200.SC_MODE_FP16}
    runs = {k: [] for k in modes}
    outs = {}
    for _ in range(a.rounds):
        for name, mode in modes.items():
            r, pri, val = leg(blob, mode, pos, moves, off, a.steps, a.warmup)
            runs[name].append(r)
            outs[name] = (pri, val)
    e = scb200.Engine(blob, 0, scb200.SC_MODE_FP32, a.leaves)
    try:
        p32, v32 = e.eval(pos, moves, off)
    finally:
        e.close()
    err = {name: {"max_abs_d_prior": float(np.abs(p - p32).max()), "max_abs_d_value": float(np.abs(v - v32).max())}
           for name, (p, v) in outs.items()}
    res = {"what": "bf16 vs fp16 tensor-core mode, 19 blocks, %d leaves, alternating engines" % a.leaves,
           "card": card(), "rounds": runs, "error_vs_fp32_engine": err}
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
