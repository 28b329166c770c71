"""Sampler time per batch with / without CUDA-graph replay.
python tools/graph_vs_stream.py [B] [H]   (each run in a fresh subprocess)"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHILD = r'''
import os, sys, torch
sys.path.insert(0, %r); sys.path.insert(0, os.path.join(%r, "oracle"))
import fdsr_oracle as O
from fastdiffsr_b200 import Engine
B, H, graph = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3] == "1"
cfg = dict(O.DEFAULT_UNET)
eng = Engine(cfg, "cuda:0", "fp16"); eng.load_state_dict(O.make_state_dict(cfg, seed=0))
eng.set_schedule(O.schedule_tables(O.make_beta_schedule(**O.DEFAULT_SCHEDULE))["betas"])
eng.set_use_graph(graph)
cond = torch.rand(B, 3, H, H, device="cuda") * 2 - 1
for i in range(3): eng.sample(cond, seed=i)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
n = 8
e0.record()
for i in range(n): eng.sample(cond, seed=i)
e1.record(); torch.cuda.synchronize()
print(e0.elapsed_time(e1) / n)
''' % (ROOT, ROOT)
B = sys.argv[1] if len(sys.argv) > 1 else "16"
H = sys.argv[2] if len(sys.argv) > 2 else "256"
for rnd in range(2):
    for graph in ("1", "0"):
        out = subprocess.run([sys.executable, "-c", CHILD, B, H, graph], capture_output=True, text=True)
        ms = out.stdout.strip().splitlines()[-1] if out.stdout.strip() else out.stderr[-300:]
        print(f"round {rnd}: graph={graph}: {ms} ms / batch (B={B}, {H}x{H})", flush=True)
