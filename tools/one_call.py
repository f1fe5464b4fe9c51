"""A few sc_eval calls of n leaves (default 1) on a 19-block bf16 engine: the command profiled for the launch lists."""
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "smart-chess-rust_b200"))
import scb200

n = int(sys.argv[1]) if len(sys.argv) > 1 else 1
mode = {"bf16": scb200.SC_MODE_BF16, "fp16": scb200.SC_MODE_FP16, "fp8": scb200.SC_MODE_FP8, "fp32": scb200.SC_MODE_FP32}[sys.argv[2] if len(sys.argv) > 2 else "bf16"]
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 6
tmp = tempfile.mkdtemp()
blob = os.path.join(tmp, "w.scw")
scb200.write_blob(scb200.random_init_state_dict(19, 0), blob)
pos, moves, off = scb200.random_positions(max(n, 4), seed=3)
e = scb200.Engine(blob, 0, mode, max(n, 16))
for _ in range(reps):
    pri, val = e.eval(pos[:n], moves[: off[n]], off[: n + 1])
print("ok", float(val[0]), e.launch_count())
e.close()
