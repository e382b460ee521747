"""Tuning aid (GPU): cfg-3 shaped Baum-Welch iteration (E-step + statistics + M-step).
usage: python tools/estep_bench.py [utts] [iters]"""
import os, sys, json
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
from sapr_b200 import _lib, engine, synth
B = int(sys.argv[1]) if len(sys.argv) > 1 else 200_000
iters = int(sys.argv[2]) if len(sys.argv) > 2 else 5
dev = torch.device("cuda", 0)
X, offsets, labels, mu, sd = synth.device_corpus(B, 11, 8, 39, 200, 20241121, dev)
A, means, var = synth.truth_models(mu, sd, 0.9)
ctx = _lib.default_context()
batch = engine.PackedBatch(X, offsets, 39, offsets.cpu().numpy(), labels)
m = engine.WordModels(11, 8, 39); m.set(means, var, A)
order = engine.group_by_model(labels)
def it():
    st, ll, _ = m.estep(batch, labels, order, engine.FP32); m.mstep(st, 1e-3); return st, ll
for _ in range(2): it()
torch.cuda.synchronize()
ctx.profile(True)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(iters): st, ll = it()
e1.record(); torch.cuda.synchronize()
k_ms, k_n = ctx.profile_read(2); s_ms, s_n = ctx.profile_read(3)
ctx.profile(False)
ms = e0.elapsed_time(e1) / iters
print(json.dumps({"utts": B, "iter_ms": ms, "estep_kernel_ms": k_ms / max(k_n, 1), "stats_kernel_ms": s_ms / max(s_n, 1),
                  "frac": 31208 * B / (ms / 1e3) / 1e9 / 6552.3, "ll_sum": float(ll.sum().item()),
                  "mean0": m.get()[0][0, 1, :3].tolist()}))
