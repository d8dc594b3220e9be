#!/usr/bin/env python3
"""rowquad (T = K C) at the C2 shape, for `ncu --set full -k regex:dgemm_kernel`."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from nonstationary_precip_b200 import ops
B, M = int(os.environ.get("B", 65536)), 1024
K = torch.randn(B, M, dtype=torch.float64, device="cuda")
C = torch.randn(M, M, dtype=torch.float64, device="cuda")
T = torch.empty_like(K)
for _ in range(3):
    ops.rowquad(K, C, T=T)
torch.cuda.synchronize()
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record(); ops.rowquad(K, C, T=T); b.record(); torch.cuda.synchronize()
print("rowquad ms", a.elapsed_time(b), "TF/s", 2 * B * M * M / a.elapsed_time(b) / 1e9)
