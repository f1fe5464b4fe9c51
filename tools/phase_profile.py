"""Debug aid: per-phase SM-cycle counters of the tcgen05 kernels (SCB200_PHASE_PROFILE=1)."""
import os, sys, tempfile
os.environ["SCB200_PHASE_PROFILE"] = "1"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "smart-chess-rust_b200"))
import bench
import numpy as np, scb200
tmp = tempfile.mkdtemp()
sd, blob = bench.make_blob(tmp, int(os.environ.get('BLOCKS', '19')))
pos, moves, off = bench.make_workload(2048, 1000)
# MODE=bf16 (default), fp16 or fp8: the operand type of the tensor-core kernels
mode = {"bf16": scb200.SC_MODE_BF16, "fp16": scb200.SC_MODE_FP16, "fp8": scb200.SC_MODE_FP8}[os.environ.get("MODE", "bf16")]
e = scb200.Engine(blob, 0, mode, 2048)
for i in range(3):
    sys.stderr.write(f"--- eval {i}\n")
    e.eval(pos, moves, off)
