"""One training-mode CIN forward + backward at the BASELINE shape: the target of `ncu --set full` captures
(5 kernels of interest: cin_tc_fwd, cin_tc_dgrad, 3 x cin_tc_wgrad).  FULL=1 selects the full saved-activation
format (bit 17 of dtb_cin_tc_set_variant) for A/B against the default compact one; PREC sets the CIN precision code;
CHECKF=1 / CHECKB=1 compare the forward / backward of that precision with the bf16x3 kernels."""
import ctypes
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deeptables_b200 import _native as nat  # noqa: E402

P = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())  # noqa: E731
B = int(os.environ.get('B', 65536))
F, D, sizes = 26, 16, (128, 128, 128)
V = 1000000
sizes_c = nat.int_array(sizes)
g = torch.Generator(device='cuda').manual_seed(0)
table = (torch.rand(F * V, D, device='cuda', generator=g) - 0.5) * 0.1
grad = torch.zeros_like(table)
offs = torch.arange(F + 1, dtype=torch.int64, device='cuda') * V
idx = torch.randint(0, V, (B, F), device='cuda', dtype=torch.int32, generator=g)
K = [26 * 26, 26 * 64, 26 * 64]
w = torch.cat([(torch.randn(k * 128, device='cuda', generator=g) / k ** 0.5) for k in K])
dw = torch.zeros_like(w)
pooled = torch.empty(B, 256, device='cuda')
d_pooled = torch.randn(B, 256, device='cuda', generator=g) * 1e-3
ws_bytes = nat.lib.dtb_cin_workspace_bytes(B, F, D, sizes_c, 3, 0, 1)
ws = torch.empty(ws_bytes, dtype=torch.uint8, device='cuda')
saved = torch.empty(nat.lib.dtb_cin_saved_bytes(B, F, D, sizes_c, 3, 0), dtype=torch.uint8, device='cuda')
prec = int(os.environ.get('PREC', 0))          # CIN precision code (4 = fp16 single pass)
nat.check(nat.lib.dtb_cin_tc_set_variant(1 | ((1 << 17) if os.environ.get('FULL') else 0)), 'cin_tc_set_variant')
reps = int(os.environ.get('REPS', 1))
for rep in range(reps):
    e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    e[0].record()
    nat.check(nat.lib.dtb_cin_fwd(P(idx), P(table), P(offs), P(w), None, P(pooled), P(saved), P(ws), ws_bytes, B, F, D,
                                  sizes_c, 3, 0, 1, prec, None, None), 'cin_fwd')
    e[1].record()
    for phase in (1, 2):                       # 1: weight pack + dgrad, 2: 3 x wgrad
        nat.check(nat.lib.dtb_cin_bwd_phase(P(idx), P(table), P(offs), P(w), P(d_pooled), P(saved), P(grad), P(dw), None,
                                            P(ws), ws_bytes, B, F, D, sizes_c, 3, 0, 1, prec, phase, None), 'cin_bwd_phase')
        e[1 + phase].record()
    torch.cuda.synchronize()
    print(f'rep {rep}: fwd {e[0].elapsed_time(e[1]):.3f} ms  dgrad {e[1].elapsed_time(e[2]):.3f} ms  wgrad '
          f'{e[2].elapsed_time(e[3]):.3f} ms  ({"full" if os.environ.get("FULL") else "compact"} saved activations, '
          f'precision {prec})', flush=True)
nat.lib.dtb_cin_tc_set_variant(1)
if os.environ.get('CHECKF'):
    # forward of this precision / kernel against the bf16x3 forward
    ref = torch.empty_like(pooled)
    nat.check(nat.lib.dtb_cin_fwd(P(idx), P(table), P(offs), P(w), None, P(ref), P(saved), P(ws), ws_bytes, B, F, D,
                                  sizes_c, 3, 0, 1, 2, None, None), 'cin_fwd ref')
    torch.cuda.synchronize()
    print(f'forward precision {prec} vs bf16x3: max err / scale {float((ref - pooled).abs().max() / ref.abs().max()):.2e}', flush=True)
if os.environ.get('CHECKB') and prec:
    # gradients of this precision's backward against the bf16x3 kernels on the same saved activations
    res = []
    nat.check(nat.lib.dtb_cin_fwd(P(idx), P(table), P(offs), P(w), None, P(pooled), P(saved), P(ws), ws_bytes, B, F, D,
                                  sizes_c, 3, 0, 1, prec, None, None), 'cin_fwd')      # ONE forward: same relu masks for both
    for pr in (2, prec):           # 2 = bf16x3 explicitly (0 = auto resolves to the fp16 kernels at this shape)
        grad.zero_()
        dw.zero_()
        for phase in (1, 2):
            nat.check(nat.lib.dtb_cin_bwd_phase(P(idx), P(table), P(offs), P(w), P(d_pooled), P(saved), P(grad), P(dw), None,
                                                P(ws), ws_bytes, B, F, D, sizes_c, 3, 0, 1, pr, phase, None), 'cin_bwd_phase')
        torch.cuda.synchronize()
        res.append((grad.clone(), dw.clone()))
    eg = float((res[0][0] - res[1][0]).abs().max() / res[0][0].abs().max())
    ew = float((res[0][1] - res[1][1]).abs().max() / res[0][1].abs().max())
    print(f'backward precision {prec} vs bf16x3: embedding grad rel err {eg:.2e}, filter grad rel err {ew:.2e}', flush=True)
