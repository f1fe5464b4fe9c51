"""sc_predict (legal moves generated on the device) against sc_eval (legal moves given by the caller) on the same leaves.

The bench.py workload (19 blocks, seed-0 net, seeded random-play leaves; ep_square recovered from each leaf's last two
history slots).  Per round the two calls alternate, each for --iters calls per size:
  * call time (host buffers in, host buffers out, the call returns after the results are in them) at n = 1 / 8 / 64;
  * leaf evals/s at n = 2048.
Then, in a pass of its own with event timing on, the legal-move kernel's device time (CUDA events on its stream) at each
size.  Before timing, sc_predict's moves are checked against the workload's host-generated moves.  Records the card name
and power limit, prints one JSON line and writes it to --out.

    python tools/predict_latency.py --out profiles/predict_latency.json
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
from bench import make_blob, make_workload  # noqa: E402

SIZES = (1, 8, 64, 2048)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def ep_from_history(pos):
    """python-chess ep_square of packed leaves: the square a double pawn push skipped, when slot 1 -> slot 0 was one."""
    ep = np.full(len(pos), -1, dtype=np.int8)
    for i, p in enumerate(pos):
        if p["n_hist"] < 2:
            continue
        mover_white = p["meta"][0] == 0
        s0, s1 = [int(x) for x in p["slot"][0]], [int(x) for x in p["slot"][1]]
        own = (lambda s: s[6]) if mover_white else (lambda s: (s[0] | s[1] | s[2] | s[3] | s[4] | s[5]) & ~s[6])
        before, after = s1[0] & own(s1), s0[0] & own(s0)
        left, arrived = before & ~after, after & ~before
        if left and arrived and not left & (left - 1) and not arrived & (arrived - 1):
            f, t = left.bit_length() - 1, arrived.bit_length() - 1
            if t - f == (16 if mover_white else -16) and f // 8 == (1 if mover_white else 6):
                ep[i] = (f + t) // 2
    return ep


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
    pos, moves, off = make_workload(2048, seed=0)
    ep = ep_from_history(pos)
    e = scb200.Engine(blob, 0, mode, 2048)
    n_max = SIZES[-1]
    out = (np.zeros((n_max, scb200.SC_MAX_MOVES), scb200.MOVE_DTYPE), np.zeros(n_max, np.int32),
           np.zeros((n_max, scb200.SC_MAX_MOVES), np.float32), np.zeros(n_max, np.float32))
    pri, val = np.zeros(int(off[-1]), np.float32), np.zeros(n_max, np.float32)

    mv, cnt, _, _ = e.predict(pos, ep, out=out)
    assert np.array_equal(cnt, np.diff(off)), "device move counts differ from the workload's"
    for i in range(n_max):
        got = mv[i, : cnt[i]]
        exp = moves[off[i] : off[i + 1]]
        assert all(np.array_equal(got[k], exp[k]) for k in ("from", "to", "promo")), i

    def call(kind, n):
        if kind == "eval":
            e.eval(pos[:n], moves[: off[n]], off[: n + 1], pri, val)
        else:
            e.predict(pos[:n], ep[:n], out=out)

    legs = {k: {n: [] for n in SIZES} for k in ("eval", "predict")}
    for n in SIZES:  # warm up every shape
        for kind in legs:
            for _ in range(5):
                call(kind, n)
    for r in range(a.rounds):
        for n in SIZES:
            iters = a.iters if n <= 64 else max(3, a.iters // 10)
            for kind in (("eval", "predict") if r % 2 == 0 else ("predict", "eval")):
                t0 = time.perf_counter()
                for _ in range(iters):
                    call(kind, n)
                legs[kind][n].append((time.perf_counter() - t0) / iters)
    e.set_timing(1)
    kernel_ms = {}
    for n in SIZES:
        t = []
        for _ in range(50):
            e.predict(pos[:n], ep[:n], out=out)
            t.append(e.predict_timing())
        kernel_ms[n] = round(statistics.median(t), 4)
    e.set_timing(0)
    e.close()

    res = {"card": card(), "mode": a.mode, "rounds": a.rounds, "leaves_with_ep": int((ep >= 0).sum()),
           "legal_moves_kernel_ms_median": kernel_ms}
    for kind, by_n in legs.items():
        r = {}
        for n in SIZES[:-1]:
            ms = [x * 1e3 for x in by_n[n]]
            r[f"call_ms_n{n}"] = {"median": round(statistics.median(ms), 4), "min": round(min(ms), 4), "max": round(max(ms), 4)}
        rate = [n_max / x for x in by_n[n_max]]
        r["leaf_evals_per_s_n2048"] = {"median": round(statistics.median(rate)), "min": round(min(rate)), "max": round(max(rate))}
        res[kind] = r
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
