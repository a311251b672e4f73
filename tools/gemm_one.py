#!/usr/bin/env python3
"""One dense GEMM shape through spfy_gemm_strided_batched, a few launches (ncu / A-B target).
    python tools/gemm_one.py m n k nb [dtype] [reps]"""
import os
import sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402
import torch
m, n, k, nb = (int(x) for x in sys.argv[1:5])
dt = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}[sys.argv[5] if len(sys.argv) > 5 else "f16"]
reps = int(sys.argv[6]) if len(sys.argv) > 6 else 5
spfy = ge.load_package()
dev = torch.device("cuda:0")
A = torch.rand(nb, m, k, device=dev).to(dt)
B = torch.rand(n, k, device=dev).to(dt)
C = torch.empty(nb, n, m, device=dev, dtype=dt)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
for _ in range(2):
    spfy.batched.gemm(A, B, C, m, n, k, transpose_a=1)
torch.cuda.synchronize()
e0.record()
for _ in range(reps):
    spfy.batched.gemm(A, B, C, m, n, k, transpose_a=1)
e1.record()
torch.cuda.synchronize()
print(f"gemm {m}x{n}x{k} nb={nb}: {e0.elapsed_time(e1) / reps * 1e3:.1f} us "
      f"(stages={os.environ.get('SPFY_GEMM_STAGES', '-')})")
