"""Time the Dense forward / backward C-ABI calls on the shapes of the bench configs (CUDA events, warm, inputs > L2).
python tools/dense_once.py  ->  one line per shape."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deeptables_b200 import _native as N  # noqa: E402

P = lambda t: None if t is None else t.data_ptr()


def timeit(fn, reps=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    shapes = [(65536 * 26, 32, 128), (65536 * 26, 128, 32), (65536, 429, 128), (65536, 128, 64), (65536, 1285, 400),
              (65536, 400, 400)]
    for rows, i, o in shapes:
        x = torch.randn(rows, i, device='cuda')
        w = torch.randn(i, o, device='cuda') / i ** 0.5
        b = torch.zeros(o, device='cuda')
        y = torch.empty(rows, o, device='cuda')
        dy = torch.randn(rows, o, device='cuda')
        dx = torch.empty(rows, i, device='cuda')
        dw = torch.zeros(i, o, device='cuda')
        db = torch.zeros(o, device='cuda')
        nb = N.lib.dtb_dense_workspace_bytes(i, o)
        ws = torch.empty(nb, dtype=torch.uint8, device='cuda')
        f = lambda: N.check(N.lib.dtb_dense_fwd(P(x), P(w), P(b), P(y), P(ws), nb, rows, i, o, 1, None), 'f')
        g = lambda: N.check(N.lib.dtb_dense_bwd(P(x), P(w), P(y), P(dy), P(dx), P(dw), P(db), P(ws), nb, rows, i, o, 1,
                                                None), 'b')
        tf, tb = timeit(f), timeit(g)
        gb_f = rows * (i + o) * 4 / 1e9
        print(f'rows {rows:8d} {i:5d} -> {o:4d}: fwd {tf:7.3f} ms ({gb_f / tf * 1e3:6.0f} GB/s algorithmic)   bwd {tb:7.3f} ms',
              flush=True)
        del x, y, dy, dx


if __name__ == '__main__':
    main()
