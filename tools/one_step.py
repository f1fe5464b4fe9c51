"""A few device-resident 2048-leaf steps on a 19-block engine (the bench.py workload): the command profiled by ncu."""
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "smart-chess-rust_b200"))
import numpy as np
import torch

import scb200

n = int(sys.argv[1]) if len(sys.argv) > 1 else 2048
mode = {"bf16": scb200.SC_MODE_BF16, "fp16": scb200.SC_MODE_FP16, "fp8": scb200.SC_MODE_FP8, "fp32": scb200.SC_MODE_FP32}[sys.argv[2] if len(sys.argv) > 2 else "bf16"]
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 4
tmp = tempfile.mkdtemp()
blob = os.path.join(tmp, "w.scw")
scb200.write_blob(scb200.random_init_state_dict(19, 0), blob)
pos, moves, off = scb200.random_positions(n, seed=1000)
e = scb200.Engine(blob, 0, mode, n)
dev = "cuda:0"
d_pos = torch.from_numpy(pos.view(np.uint8)).to(dev)
d_moves = torch.from_numpy(moves.view(np.uint8)).to(dev)
d_off = torch.from_numpy(off).to(dev)
d_pri = torch.zeros(int(off[n]), dtype=torch.float32, device=dev)
d_val = torch.zeros(n, dtype=torch.float32, device=dev)
st = torch.cuda.Stream()
for _ in range(reps):
    e.eval_device(n, d_pos, d_moves, d_off, int(off[n]), d_pri, d_val, st.cuda_stream)
st.synchronize()
print("ok", float(d_val[0]), e.launch_count())
e.close()
