"""Timing of the in-flight batch (tnb_ttsvd_batch): prints ms per tensor for the 64^5 / r=32 workload with `inflight`
tensors in flight and `reserve` SMs left free by the whole-GPU kernels.  Usage: batch_exp.py [inflight] [reserve]"""
import sys

import torch

sys.path.insert(0, ".")
from tntorch_b200 import ops

B = int(sys.argv[1]) if len(sys.argv) > 1 else 6
reserve = int(sys.argv[2]) if len(sys.argv) > 2 else 4
shape = (64,) * 5
ops.set_reserved_sms(reserve)
X = torch.empty((B,) + shape, device="cuda")
for b in range(B):
    X[b].normal_()
plan = ops.TTSVDBatchPlan(shape, torch.float32, B, rmax=32, inflight=B)
for _ in range(2):
    plan.run(X)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
K = 5
for _ in range(K):
    plan.run(X)
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / K
print(f"inflight={B} reserve={reserve}: {ms:.2f} ms per batch, {ms / B:.2f} ms per tensor, {B * 2**30 / ms / 1e6:.1f} GElements/s, spec={list(plan.spec)}")
