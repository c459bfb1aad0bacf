"""Time the bf16x3 and bf16x1 CIN forward at the BASELINE shape (B=65536, 26x16, CIN 128x128x128)."""
import ctypes
import os
import sys
import numpy as np
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deeptables_b200 import _native as nat

P = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())
B = int(os.environ.get('B', 65536))
F, D, sizes = 26, 16, (128, 128, 128)
V = 100000
sizes_c = nat.int_array(sizes)
g = torch.Generator(device='cuda').manual_seed(0)
table = (torch.rand(F * V, D, device='cuda', generator=g) - 0.5) * 0.1
offs = torch.arange(F + 1, dtype=torch.int64, device='cuda') * V
idx = torch.randint(0, V, (B, F), device='cuda', dtype=torch.int32, generator=g)
K = [26 * 26, 26 * 64, 26 * 64]
w = torch.cat([(torch.randn(k * 128, device='cuda', generator=g) / k ** 0.5) for k in K])
pooled = torch.empty(B, 256, device='cuda')
ws_bytes = nat.lib.dtb_cin_workspace_bytes(B, F, D, sizes_c, 3, 0, 1)
ws = torch.empty(ws_bytes, dtype=torch.uint8, device='cuda')
saved = torch.empty(nat.lib.dtb_cin_saved_bytes(B, F, D, sizes_c, 3, 0), dtype=torch.uint8, device='cuda')
flop = B * 2 * D * 128 * sum(K)


def run(precision, train):
    nat.check(nat.lib.dtb_cin_fwd(P(idx), P(table), P(offs), P(w), None, P(pooled), P(saved) if train else None, P(ws),
                                  ws_bytes, B, F, D, sizes_c, 3, 0, 1, precision, None, None))


only = os.environ.get('ONLY')
for precision in (2, 3):
    for train in (0,):
        tag = f'pass={"bf16x3" if precision == 2 else "bf16x1"} train={train}'
        if only and only != f'{precision}{train}':
            continue
        for _ in range(2):
            run(precision, train)
        torch.cuda.synchronize()
        ts = []
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); run(precision, train); e1.record(); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        t = sorted(ts)[2]
        print(f'{tag}: {t:.3f} ms  algorithmic {flop / t / 1e9:.0f} TFLOP/s', flush=True)
