"""GPU parity tests: every C-ABI op against the CPU oracle on the same seeded inputs.
fp32 kernels: rtol 1e-4 (tolerance stated per test); index bookkeeping bit-exact."""
import ctypes

import os

import numpy as np
import pytest
import torch

from oracle import layers_ref as L

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def nat():
    from deeptables_b200 import _native
    return _native


_KEEP = []     # ctypes only sees raw pointers: keep every device tensor of a test alive until it ends


@pytest.fixture(autouse=True)
def _keepalive():
    _KEEP.clear()
    yield
    torch.cuda.synchronize()
    _KEEP.clear()


def dev(a, dtype=None):
    t = torch.as_tensor(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    t = t.cuda()
    _KEEP.append(t)
    return t


def make_table(vocab, d, seed=0):
    g = np.random.default_rng(seed)
    tabs = [g.uniform(-0.5, 0.5, size=(v, d)).astype(np.float32) for v in vocab]
    offs = np.concatenate([[0], np.cumsum(vocab)]).astype(np.int64)
    return tabs, np.concatenate(tabs, axis=0), offs


def make_idx(vocab, b, seed=1):
    g = np.random.default_rng(seed)
    return np.stack([g.integers(0, v, size=b) for v in vocab], axis=1).astype(np.int32)


def P(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


SHAPES = [  # (vocab sizes, D, C, B)
    ([50] * 26, 16, 13, 257),     # Criteo shape
    ([7, 5, 9, 4], 4, 3, 64),     # README-like small dims
    ([11, 3], 2, 0, 33),          # D=2: generic (non-vector) path, no continuous
    ([13], 8, 2, 19),             # single categorical column
    ([6, 7, 8], 32, 1, 40),       # D=32
]


@pytest.mark.parametrize('vocab,d,c,b', SHAPES)
def test_gather_scatter_bit_exact(nat, vocab, d, c, b):
    tabs, flat, offs = make_table(vocab, d)
    idx = make_idx(vocab, b)
    f = len(vocab)
    out = torch.empty(b, f, d, device='cuda')
    status = torch.zeros(1, dtype=torch.int32, device='cuda')
    nat.check(nat.lib.dtb_embedding_gather(P(dev(idx)), P(dev(flat)), P(dev(offs)), P(out), b, f, d, P(status), None))
    want = torch.cat(L.embedding_lookup([torch.tensor(t) for t in tabs], torch.tensor(idx)), dim=1)
    assert torch.equal(out.cpu(), want)            # pure data movement: bit exact
    assert int(status.item()) == 0
    # scatter-add == gradient of the gather (duplicates accumulate)
    gout = np.random.default_rng(3).normal(size=(b, f, d)).astype(np.float32)
    gt = torch.zeros(flat.shape, device='cuda')
    nat.check(nat.lib.dtb_embedding_scatter_add(P(dev(idx)), P(dev(offs)), P(dev(gout)), P(gt), b, f, d, None))
    want_g = np.zeros_like(flat, dtype=np.float64)
    for i in range(f):
        np.add.at(want_g, offs[i] + idx[:, i], gout[:, i].astype(np.float64))
    np.testing.assert_allclose(gt.cpu().numpy(), want_g, rtol=1e-5, atol=1e-6)


def test_out_of_range_id_sets_status_and_reads_zero(nat):
    vocab, d, b = [5, 6], 4, 3
    _, flat, offs = make_table(vocab, d)
    idx = np.array([[1, 2], [5, 0], [0, -1]], dtype=np.int32)      # (1,0) and (2,1) invalid
    out = torch.full((b, 2, d), 7.0, device='cuda')
    status = torch.zeros(1, dtype=torch.int32, device='cuda')
    nat.check(nat.lib.dtb_embedding_gather(P(dev(idx)), P(dev(flat)), P(dev(offs)), P(out), b, 2, d, P(status), None))
    assert int(status.item()) == 0b11
    assert float(out[1, 0].abs().sum()) == 0.0 and float(out[2, 1].abs().sum()) == 0.0
    assert float(out[0].abs().sum()) > 0


@pytest.mark.parametrize('vocab,d,c,b', SHAPES)
def test_fm_linear_fwd_bwd(nat, vocab, d, c, b):
    tabs, flat, offs = make_table(vocab, d)
    idx = make_idx(vocab, b)
    f = len(vocab)
    g = np.random.default_rng(5)
    dense = g.normal(size=(b, c)).astype(np.float32) if c else None
    wl = g.normal(size=(f + c,)).astype(np.float32)
    d_idx, d_tab, d_offs = dev(idx), dev(flat), dev(offs)
    d_dense = dev(dense) if c else None
    d_wl = dev(wl)
    out_lin = torch.empty(b, device='cuda')
    out_fm = torch.empty(b, device='cuda')
    nat.check(nat.lib.dtb_fm_linear_fwd(P(d_idx), P(d_tab), P(d_offs), P(d_dense), P(d_wl), P(out_lin), P(out_fm),
                                        b, f, d, c, None, None))
    # oracle (float64 for a tight check)
    t64 = [torch.tensor(t, dtype=torch.float64, requires_grad=True) for t in tabs]
    emb = L.embedding_lookup(t64, torch.tensor(idx))
    dn = torch.tensor(dense, dtype=torch.float64) if c else None
    w64 = torch.tensor(wl, dtype=torch.float64, requires_grad=True)
    lin = L.linear(emb, dn, w64.reshape(-1, 1))
    fm = L.fm(L.concat_embeddings(emb))
    np.testing.assert_allclose(out_lin.cpu().numpy(), lin.detach().numpy()[:, 0], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(out_fm.cpu().numpy(), fm.detach().numpy()[:, 0], rtol=1e-4, atol=1e-5)
    # backward
    g_lin = g.normal(size=b).astype(np.float32)
    g_fm = g.normal(size=b).astype(np.float32)
    gt = torch.zeros(flat.shape, device='cuda')
    gw = torch.zeros(f + c, device='cuda')
    nat.check(nat.lib.dtb_fm_linear_bwd(P(d_idx), P(d_tab), P(d_offs), P(d_dense), P(d_wl), P(dev(g_lin)),
                                        P(dev(g_fm)), P(gt), P(gw), b, f, d, c, None))
    loss = (lin[:, 0] * torch.tensor(g_lin, dtype=torch.float64)).sum() + \
           (fm[:, 0] * torch.tensor(g_fm, dtype=torch.float64)).sum()
    grads = torch.autograd.grad(loss, t64 + [w64])
    want_t = torch.cat(grads[:-1], dim=0).numpy()
    np.testing.assert_allclose(gt.cpu().numpy(), want_t, rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(gw.cpu().numpy(), grads[-1].numpy(), rtol=1e-4, atol=1e-4)
    # FM only / linear only branches
    out2 = torch.empty(b, device='cuda')
    nat.check(nat.lib.dtb_fm_linear_fwd(P(d_idx), P(d_tab), P(d_offs), None, None, None, P(out2), b, f, d, 0, None, None))
    np.testing.assert_allclose(out2.cpu().numpy(), fm.detach().numpy()[:, 0], rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize('vocab,d,c,b', SHAPES)
def test_concat_and_batchnorm(nat, vocab, d, c, b):
    tabs, flat, offs = make_table(vocab, d)
    idx = make_idx(vocab, b)
    f = len(vocab)
    w = f * d + c
    g = np.random.default_rng(6)
    dense = (g.normal(size=(b, c)) * 3 + 1).astype(np.float32) if c else None
    X = torch.empty(b, w, device='cuda')
    nat.check(nat.lib.dtb_concat_emb_dense_fwd(P(dev(idx)), P(dev(flat)), P(dev(offs)), P(dev(dense)) if c else None,
                                               P(X), b, f, d, c, None, None))
    emb = L.embedding_lookup([torch.tensor(t) for t in tabs], torch.tensor(idx))
    want = L.flatten_embeddings(emb)
    if c:
        want = torch.cat([want, torch.tensor(dense)], dim=-1)
    assert torch.equal(X.cpu(), want)              # data movement: bit exact, field-major layout
    gamma = (g.normal(size=w) + 2).astype(np.float32)
    beta = g.normal(size=w).astype(np.float32)
    mm = torch.zeros(w, device='cuda')
    mv = torch.ones(w, device='cuda')
    sm, sv = torch.empty(w, device='cuda'), torch.empty(w, device='cuda')
    ws = torch.empty(2 * w, dtype=torch.float64, device='cuda')
    Y = torch.empty_like(X)
    d_g, d_b = dev(gamma), dev(beta)
    nat.check(nat.lib.dtb_batchnorm_train_fwd(P(X), P(Y), P(d_g), P(d_b), P(mm), P(mv), P(sm), P(sv), P(ws), b, w,
                                              1e-3, 0.99, None))
    x64 = want.double().requires_grad_(True)
    g64 = torch.tensor(gamma, dtype=torch.float64, requires_grad=True)
    b64 = torch.tensor(beta, dtype=torch.float64, requires_grad=True)
    y64, nm, nv = L.batch_norm(x64, g64, b64, torch.zeros(w, dtype=torch.float64),
                               torch.ones(w, dtype=torch.float64), True)
    np.testing.assert_allclose(Y.cpu().numpy(), y64.detach().numpy(), rtol=1e-4, atol=2e-5)
    np.testing.assert_allclose(mm.cpu().numpy(), nm.numpy(), rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(mv.cpu().numpy(), nv.numpy(), rtol=1e-5, atol=1e-7)
    dy = g.normal(size=(b, w)).astype(np.float32)
    dX = torch.empty_like(X)
    dg, db = torch.zeros(w, device='cuda'), torch.zeros(w, device='cuda')
    nat.check(nat.lib.dtb_batchnorm_bwd(P(X), P(dev(dy)), P(dX), P(d_g), P(sm), P(sv), P(dg), P(db), P(ws), b, w,
                                        1e-3, None))
    gx, gg, gb = torch.autograd.grad((y64 * torch.tensor(dy, dtype=torch.float64)).sum(), [x64, g64, b64])
    np.testing.assert_allclose(dX.cpu().numpy(), gx.numpy(), rtol=1e-3, atol=2e-5)
    np.testing.assert_allclose(dg.cpu().numpy(), gg.numpy(), rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(db.cpu().numpy(), gb.numpy(), rtol=1e-4, atol=1e-4)
    # inference mode with the moving statistics
    Y2 = torch.empty_like(X)
    nat.check(nat.lib.dtb_batchnorm_infer_fwd(P(X), P(Y2), P(d_g), P(d_b), P(mm), P(mv), b, w, 1e-3, None))
    y2, _, _ = L.batch_norm(want.double(), g64.detach(), b64.detach(), nm, nv, False)
    np.testing.assert_allclose(Y2.cpu().numpy(), y2.numpy(), rtol=1e-4, atol=2e-5)
    # concat backward scatters only the embedding columns
    gt = torch.zeros(flat.shape, device='cuda')
    nat.check(nat.lib.dtb_concat_emb_dense_bwd(P(dev(idx)), P(dev(offs)), P(dev(dy)), P(gt), b, f, d, c, None))
    want_g = np.zeros(flat.shape, dtype=np.float64)
    for i in range(f):
        np.add.at(want_g, offs[i] + idx[:, i], dy[:, i * d:(i + 1) * d].astype(np.float64))
    np.testing.assert_allclose(gt.cpu().numpy(), want_g, rtol=1e-5, atol=1e-6)


# wide layers = tcgen05 GEMMs (dense_tc.cu): tower shapes, 1079-wide PNN input, AutoInt projection (32 -> 128), ragged
# row counts / odd widths, more than one 256-column output tile (dX of the 1079-wide layer), K smaller than one chunk
@pytest.mark.parametrize('rows,i,o,act', [(300, 429, 128, 1), (300, 128, 64, 1), (77, 64, 1, 0), (50, 1, 1, 0),
                                           (64, 37, 3, 0), (5, 10, 20, 1), (1000, 1079, 128, 1), (2600, 32, 128, 1),
                                           (129, 845, 128, 0), (33, 7, 300, 1), (4097, 64, 64, 0)])
def test_dense_fwd_bwd(nat, rows, i, o, act):
    g = np.random.default_rng(7)
    x = g.normal(size=(rows, i)).astype(np.float32)
    w = (g.normal(size=(i, o)) / np.sqrt(i)).astype(np.float32)
    bias = g.normal(size=o).astype(np.float32)
    dy = g.normal(size=(rows, o)).astype(np.float32)
    X, W, Bv = dev(x), dev(w), dev(bias)
    Y = torch.empty(rows, o, device='cuda')
    wsb = nat.lib.dtb_dense_workspace_bytes(i, o)
    ws = torch.empty(max(wsb, 16), dtype=torch.uint8, device='cuda')
    nat.check(nat.lib.dtb_dense_fwd(P(X), P(W), P(Bv), P(Y), P(ws), wsb, rows, i, o, act, None))
    x64 = torch.tensor(x, dtype=torch.float64, requires_grad=True)
    w64 = torch.tensor(w, dtype=torch.float64, requires_grad=True)
    b64 = torch.tensor(bias, dtype=torch.float64, requires_grad=True)
    y64 = L.dense(x64, w64, b64, 'relu' if act else None)
    # out_dim > 8: tcgen05 GEMM on bf16 hi/lo splits (three passes, the dropped lo*lo term is 2^-16 of a product): a
    # few 1e-5 absolute on O(1) outputs; the narrow kernels are plain fp32
    tc = o > 8
    np.testing.assert_allclose(Y.cpu().numpy(), y64.detach().numpy(), rtol=1e-4, atol=1e-4 if tc else 1e-5)
    dY = dev(dy)
    dX = torch.empty(rows, i, device='cuda')
    dW = torch.zeros(i, o, device='cuda')
    dB = torch.zeros(o, device='cuda')
    # the backward takes the relu mask from Y: hand it the oracle's Y, otherwise an output whose pre-activation lies within
    # the forward's rounding error of zero flips its mask bit and a whole row of dX moves by |dy . W| (seen on the B200
    # at 128 000+ outputs: one such element) -- that is the forward's tolerance, not the backward's arithmetic
    Yb = dev(y64.detach().numpy().astype(np.float32))
    nat.check(nat.lib.dtb_dense_bwd(P(X), P(W), P(Yb), P(dY), P(dX), P(dW), P(dB), P(ws), wsb, rows, i, o, act, None))
    gx, gw, gb = torch.autograd.grad((y64 * torch.tensor(dy, dtype=torch.float64)).sum(), [x64, w64, b64])
    np.testing.assert_allclose(dX.cpu().numpy(), gx.numpy(), rtol=1e-4, atol=1e-4 if tc else 1e-5)
    wsc = max(1.0, float(gw.abs().max()))
    np.testing.assert_allclose(dW.cpu().numpy(), gw.numpy(), rtol=1e-4, atol=(1e-4 * wsc) if tc else 1e-4)
    np.testing.assert_allclose(dB.cpu().numpy(), gb.numpy(), rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize('task,cols', [(0, 1), (0, 3), (1, 1), (2, 4)])
def test_losses(nat, task, cols):
    g = np.random.default_rng(8)
    rows = 130
    z = (g.normal(size=(rows, cols)) * 2).astype(np.float32)
    if task == 0:
        y = (g.random((rows, cols)) < 0.4).astype(np.float32)
    elif task == 1:
        y = g.normal(size=(rows, cols)).astype(np.float32)
    else:
        y = np.eye(cols, dtype=np.float32)[g.integers(0, cols, size=rows)]
    sw = g.uniform(0.5, 2.0, size=rows).astype(np.float32)
    for weights in (None, sw):
        prob = torch.empty(rows, cols, device='cuda')
        dz = torch.empty(rows, cols, device='cuda')
        acc = torch.zeros(1, dtype=torch.float64, device='cuda')
        nat.check(nat.lib.dtb_loss_fwd_bwd(P(dev(z)), P(dev(y)), P(dev(weights)) if weights is not None else None,
                                           P(prob), P(dz), P(acc), rows, cols, task, None))
        z64 = torch.tensor(z, dtype=torch.float64, requires_grad=True)
        y64 = torch.tensor(y, dtype=torch.float64)
        if task == 0:
            p = torch.sigmoid(z64)
            per = -(y64 * torch.log(p.clamp(1e-7, 1 - 1e-7)) + (1 - y64) * torch.log((1 - p).clamp(1e-7, 1))).mean(-1)
        elif task == 1:
            p = z64
            per = ((p - y64) ** 2).mean(-1)
        else:
            p = torch.softmax(z64, -1)
            per = -(y64 * torch.log(p.clamp(1e-7, 1 - 1e-7))).sum(-1)
        wv = torch.tensor(weights, dtype=torch.float64) if weights is not None else torch.ones(rows, dtype=torch.float64)
        loss = (per * wv).sum() / rows
        (gz,) = torch.autograd.grad(loss, [z64])
        np.testing.assert_allclose(prob.cpu().numpy(), p.detach().numpy(), rtol=1e-4, atol=1e-6)
        np.testing.assert_allclose(dz.cpu().numpy(), gz.numpy(), rtol=2e-4, atol=1e-7)
        np.testing.assert_allclose(float(acc.item()) / rows, float(loss), rtol=1e-5)


def test_adam_dense_matches_oracle(nat):
    g = np.random.default_rng(9)
    n = 1000
    p0 = g.normal(size=n).astype(np.float32)
    pt, m, v = dev(p0.copy()), torch.zeros(n, device='cuda'), torch.zeros(n, device='cuda')
    po, mo, vo = torch.tensor(p0.copy()), torch.zeros(n), torch.zeros(n)
    from deeptables_b200.engine import adam_alpha
    for step in range(1, 6):
        grad = g.normal(size=n).astype(np.float32)
        gd = dev(grad.copy())
        nat.check(nat.lib.dtb_adam_dense(P(pt), P(m), P(v), P(gd), n, adam_alpha(step), 0.9, 0.999, 1e-7, 1, None))
        assert float(gd.abs().sum()) == 0.0                   # zero_grad
        L.adam_step(po, torch.tensor(grad), mo, vo, step)
    # the kernel pins m/v with fused multiply-adds, torch-CPU rounds twice: allow a few ulps
    np.testing.assert_allclose(pt.cpu().numpy(), po.numpy(), rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(m.cpu().numpy(), mo.numpy(), rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(v.cpu().numpy(), vo.numpy(), rtol=1e-5, atol=1e-9)


def test_lazy_adam_matches_dense(nat):
    """Exact-lazy row-wise Adam is BIT-identical to dense Adam over the whole table."""
    from deeptables_b200.engine import adam_alpha
    vocab, d, b, steps = [40, 25, 60], 16, 12, 25
    f = len(vocab)
    rows = sum(vocab)
    offs = dev(np.concatenate([[0], np.cumsum(vocab)]).astype(np.int64))
    g = np.random.default_rng(10)
    w0 = g.uniform(-0.05, 0.05, size=(rows, d)).astype(np.float32)
    alpha = dev(np.array([0.0] + [adam_alpha(s) for s in range(1, steps + 2)], dtype=np.float32))
    wd, md, vd = dev(w0.copy()), torch.zeros(rows, d, device='cuda'), torch.zeros(rows, d, device='cuda')
    wl, ml, vl = dev(w0.copy()), torch.zeros(rows, d, device='cuda'), torch.zeros(rows, d, device='cuda')
    gl = torch.zeros(rows, d, device='cuda')
    last = torch.zeros(rows, dtype=torch.int32, device='cuda')
    for step in range(1, steps + 1):
        idx = make_idx(vocab, b, seed=100 + step)
        idx[1] = idx[0]                                            # duplicate ids inside a batch
        d_idx = dev(idx)
        nat.check(nat.lib.dtb_adam_rows_catchup(P(d_idx), P(offs), P(wl), P(ml), P(vl), P(last), P(alpha), step - 1,
                                                0.9, 0.999, 1e-7, b, f, d, None))
        # rows read by this step must already equal the dense trajectory
        flat_rows = (offs[:-1].cpu().numpy()[None, :] + idx).reshape(-1)
        assert torch.equal(wl[flat_rows], wd[flat_rows])
        gout = g.normal(size=(b, f, d)).astype(np.float32)
        gd = torch.zeros(rows, d, device='cuda')
        nat.check(nat.lib.dtb_embedding_scatter_add(P(d_idx), P(offs), P(dev(gout)), P(gd), b, f, d, None))
        gl.copy_(gd)        # identical gradient bits for both optimisers (atomic order is not deterministic)
        a = float(alpha[step].item())
        nat.check(nat.lib.dtb_adam_dense(P(wd), P(md), P(vd), P(gd), rows * d, a, 0.9, 0.999, 1e-7, 1, None))
        nat.check(nat.lib.dtb_adam_rows_apply(P(d_idx), P(offs), P(wl), P(ml), P(vl), P(gl), P(last), P(alpha), step,
                                              0.9, 0.999, 1e-7, b, f, d, None))
        assert float(gl.abs().sum()) == 0.0
    nat.check(nat.lib.dtb_adam_rows_flush(P(wl), P(ml), P(vl), P(last), P(alpha), steps, 0.9, 0.999, 1e-7, rows, d, None))
    assert torch.equal(wl, wd) and torch.equal(ml, md) and torch.equal(vl, vd)
    assert int(last.min().item()) == steps


def test_lazy_adam_long_gap_is_bit_exact_and_bounded(nat):
    """A row untouched for thousands of steps (rare id of a long-tailed column): the replay leaves the full update
    once m has reached the fixed point of its decay and finishes with the v-only tail -- still the dense kernel's bits."""
    from deeptables_b200.engine import adam_alpha
    rows, d, gap = 64, 16, 6000
    g = np.random.default_rng(3)
    w0 = g.uniform(-0.05, 0.05, size=(rows, d)).astype(np.float32)
    g0 = g.normal(size=(rows, d)).astype(np.float32) * np.logspace(-6, 0, rows, dtype=np.float32)[:, None]
    alpha = dev(np.array([0.0] + [adam_alpha(s) for s in range(1, gap + 3)], dtype=np.float32))
    offs = dev(np.array([0, rows], dtype=np.int64))
    ids = dev(np.arange(rows, dtype=np.int32).reshape(rows, 1))
    wd, md, vd, gd = dev(w0.copy()), torch.zeros(rows, d, device='cuda'), torch.zeros(rows, d, device='cuda'), dev(g0.copy())
    wl, ml, vl, gl = dev(w0.copy()), torch.zeros(rows, d, device='cuda'), torch.zeros(rows, d, device='cuda'), dev(g0.copy())
    last = torch.zeros(rows, dtype=torch.int32, device='cuda')
    nat.check(nat.lib.dtb_adam_rows_apply(P(ids), P(offs), P(wl), P(ml), P(vl), P(gl), P(last), P(alpha), 1, 0.9, 0.999,
                                          1e-7, rows, 1, d, None))
    for step in range(1, gap + 1):          # dense: the gradient step, then gap-1 zero-gradient steps
        nat.check(nat.lib.dtb_adam_dense(P(wd), P(md), P(vd), P(gd), rows * d, float(alpha[step].item()), 0.9, 0.999,
                                         1e-7, 1, None))
    nat.check(nat.lib.dtb_adam_rows_catchup(P(ids), P(offs), P(wl), P(ml), P(vl), P(last), P(alpha), gap, 0.9, 0.999, 1e-7,
                                            rows, 1, d, None))
    for name, a_, b_ in (('weights', wl, wd), ('m', ml, md), ('v', vl, vd)):
        bad = (a_ != b_)
        assert not bool(bad.any()), (f'{name}: {int(bad.sum())} of {bad.numel()} entries differ, max |diff| '
                                     f'{float((a_ - b_).abs().max()):.3e}, first at {bad.nonzero()[0].tolist()}: '
                                     f'lazy {float(a_[bad][0]):.9e} dense {float(b_[bad][0]):.9e}')
    assert float(md.abs().max()) < 1e-44          # the gap really is past the decay of m


CIN_CASES = [  # (F, D, sizes, direct, bias, act)
    (5, 4, (6, 4), False, False, 1),
    (26, 16, (32, 32, 16), False, False, 1),
    (4, 8, (6, 5), True, True, 1),
    (3, 2, (4, 3), False, True, 0),
    (1, 4, (4, 2), False, False, 1),
    (7, 32, (8,), False, False, 1),
]


def _cin_oracle(x, sizes, direct, filters, biases, act):
    params = dict(cross_layer_size=sizes, direct=direct, use_bias=biases is not None,
                  activation='relu' if act else 'linear')
    width = L.cin_pooled_width(x.shape[1], params)
    w = {f'f_{k}': filters[k].unsqueeze(0) for k in range(len(sizes))}
    if biases is not None:
        for k in range(len(sizes)):
            w[f'bias{k}'] = biases[k]
    # identity head so that the oracle returns the pooled features column by column
    outs = []
    for col in range(width):
        kernel = torch.zeros(width, 1, dtype=x.dtype)
        kernel[col, 0] = 1.0
        w['exFM_out/kernel'] = kernel
        w['exFM_out/bias'] = torch.zeros(1, dtype=x.dtype)
        outs.append(L.cin(x, params, w))
    return torch.cat(outs, dim=1)


@pytest.mark.parametrize('f,d,sizes,direct,use_bias,act', CIN_CASES)
@pytest.mark.parametrize('precision', [1, 2, 0])
def test_cin_fwd_bwd(nat, f, d, sizes, direct, use_bias, act, precision):
    """precision 1 = any-shape formulation, 2 = tensor-core bf16x3 (skipped where the shape is outside it), 0 = auto:
    the single-pass fp16 kernels where they apply (error ~2e-4 of the scale).  Under fp16 a pre-activation within that
    error of zero can flip its relu-mask bit against the float64 oracle, which moves the gradient rows of that one batch
    row by percents: the gradient check then asks for 99 % of the entries inside the tolerance and a small norm-wise
    error (95 % / 5e-2 at these 37 rows); the backward ARITHMETIC of the fp16 kernels is checked against the bf16x3 kernels on identical activations in
    tests/test_zz_baseline_configs_gpu.py."""
    b = 37
    vocab = [9 + i for i in range(f)]
    tabs, flat, offs = make_table(vocab, d, seed=11)
    idx = make_idx(vocab, b, seed=12)
    g = np.random.default_rng(13)
    fns = L.cin_field_nums(f, sizes, direct)
    filt = [(g.normal(size=(f * fns[k], s)) / np.sqrt(f * fns[k])).astype(np.float32) for k, s in enumerate(sizes)]
    bias = [g.normal(size=s).astype(np.float32) * 0.1 for s in sizes] if use_bias else None
    wcat = np.concatenate([x.reshape(-1) for x in filt])
    sizes_c = nat.int_array(sizes)
    n = len(sizes)
    if precision == 2 and not nat.lib.dtb_cin_tc_supported(f, d, sizes_c, n, int(direct)):
        pytest.skip('shape outside the tensor-core kernels')
    pw = L.cin_pooled_width(f, dict(cross_layer_size=sizes, direct=direct))
    pooled = torch.empty(b, pw, device='cuda')
    ws_bytes = nat.lib.dtb_cin_workspace_bytes(b, f, d, sizes_c, n, int(direct), 1)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device='cuda')
    saved = torch.empty(nat.lib.dtb_cin_saved_bytes(b, f, d, sizes_c, n, int(direct)), dtype=torch.uint8, device='cuda')
    d_idx, d_tab, d_offs, d_w = dev(idx), dev(flat), dev(offs), dev(wcat)
    d_b = dev(np.concatenate(bias)) if use_bias else None
    nat.check(nat.lib.dtb_cin_fwd(P(d_idx), P(d_tab), P(d_offs), P(d_w), P(d_b), P(pooled), P(saved), P(ws), ws_bytes,
                                  b, f, d, sizes_c, n, int(direct), act, precision, None, None))
    t64 = [torch.tensor(t, dtype=torch.float64, requires_grad=True) for t in tabs]
    x = torch.cat(L.embedding_lookup(t64, torch.tensor(idx)), dim=1)
    f64 = [torch.tensor(w_, dtype=torch.float64, requires_grad=True) for w_ in filt]
    b64 = [torch.tensor(b_, dtype=torch.float64, requires_grad=True) for b_ in bias] if use_bias else None
    want = _cin_oracle(x, sizes, direct, f64, b64, act)
    scale = float(want.abs().max())
    tol = 1e-4 if precision == 1 else 1e-3            # fp32 path vs bf16x3 tensor-core path
    np.testing.assert_allclose(pooled.cpu().numpy(), want.detach().numpy(), rtol=tol, atol=tol * scale)
    dp = g.normal(size=(b, pw)).astype(np.float32)
    gt = torch.zeros(flat.shape, device='cuda')
    dw = torch.zeros(wcat.shape, device='cuda')
    dbias = torch.zeros(sum(sizes), device='cuda') if use_bias else None
    nat.check(nat.lib.dtb_cin_bwd(P(d_idx), P(d_tab), P(d_offs), P(d_w), P(dev(dp)), P(saved), P(gt), P(dw), P(dbias),
                                  P(ws), ws_bytes, b, f, d, sizes_c, n, int(direct), act, precision, None))
    loss = (want * torch.tensor(dp, dtype=torch.float64)).sum()
    params = t64 + f64 + (b64 or [])
    grads = torch.autograd.grad(loss, params, allow_unused=True)
    want_t = torch.cat(grads[:f], dim=0).numpy()
    want_w = np.concatenate([gg.numpy().reshape(-1) for gg in grads[f:f + n]])
    def close(got, want_, what):
        got = got.cpu().numpy()
        if precision != 0:
            np.testing.assert_allclose(got, want_, rtol=tol * 10, atol=tol * np.abs(want_).max(), err_msg=what)
            return
        ok = np.abs(got - want_) <= tol * 10 * np.abs(want_) + tol * np.abs(want_).max()
        # 37 batch rows: ONE flipped mask bit moves that row's share of every filter entry
        assert ok.mean() >= 0.95, f'{what}: only {100 * ok.mean():.2f} % of the entries inside the tolerance'
        rel = np.linalg.norm(got - want_) / np.linalg.norm(want_)
        assert rel <= 5e-2, f'{what}: norm-wise error {rel:.2e}'

    close(gt, want_t, 'embedding gradient')
    close(dw, want_w, 'filter gradient')
    if use_bias:
        close(dbias, np.concatenate([gg.numpy() for gg in grads[f + n:]]), 'bias gradient')


def test_cin_invalid_config_rejected(nat):
    sizes_c = nat.int_array((3, 4))
    assert nat.lib.dtb_cin_workspace_bytes(4, 3, 4, sizes_c, 2, 0, 1) == 0      # odd non-last layer, direct=False
    dummy = torch.zeros(16, device='cuda')
    rc = nat.lib.dtb_cin_fwd(P(dummy), P(dummy), P(dummy), P(dummy), None, P(dummy), None, P(dummy), 64, 4, 3, 4,
                             sizes_c, 2, 0, 1, 1, None, None)
    assert rc == -1 and 'cross_layer_size' in nat.last_error()


# (70, 845, 6) = BASELINE configs[3] (F*32 + 13), (40, 1079, 4) PNN-width, (21, 1500, 3) shared-memory kernels,
# (30, 300, 10) more layers than one reduction launch holds
@pytest.mark.parametrize('b,w,n', [(50, 429, 6), (33, 17, 1), (64, 40, 4), (70, 845, 6), (40, 1079, 4), (21, 1500, 3),
                                   (30, 300, 10)])
def test_cross_fwd_bwd(nat, b, w, n):
    g = np.random.default_rng(14)
    x = g.normal(size=(b, w)).astype(np.float32)
    ks = (g.normal(size=(n, w)) / np.sqrt(w)).astype(np.float32)
    bs = (g.normal(size=(n, w)) * 0.1).astype(np.float32)
    X, K, Bv = dev(x), dev(ks), dev(bs)
    Y = torch.empty(b, w, device='cuda')
    xw = torch.empty(b, n, device='cuda')
    nat.check(nat.lib.dtb_cross_fwd(P(X), P(K), P(Bv), P(Y), P(xw), b, w, n, None))
    x64 = torch.tensor(x, dtype=torch.float64, requires_grad=True)
    k64 = [torch.tensor(ks[i].reshape(w, 1), dtype=torch.float64, requires_grad=True) for i in range(n)]
    b64 = [torch.tensor(bs[i].reshape(w, 1), dtype=torch.float64, requires_grad=True) for i in range(n)]
    y64 = L.cross(x64, k64, b64)
    np.testing.assert_allclose(Y.cpu().numpy(), y64.detach().numpy(), rtol=1e-4, atol=1e-4)
    dy = g.normal(size=(b, w)).astype(np.float32)
    dX = torch.empty(b, w, device='cuda')
    dK, dB = torch.zeros(n, w, device='cuda'), torch.zeros(n, w, device='cuda')
    wsb = nat.lib.dtb_cross_bwd_workspace_bytes(b, w, n)
    wsc = torch.empty(wsb, dtype=torch.uint8, device='cuda')
    nat.check(nat.lib.dtb_cross_bwd(P(X), P(K), P(Bv), P(xw), P(dev(dy)), P(dX), P(dK), P(dB), P(wsc), wsb, b, w, n, None))
    grads = torch.autograd.grad((y64 * torch.tensor(dy, dtype=torch.float64)).sum(), [x64] + k64 + b64)
    sc = max(1.0, float(grads[0].abs().max()))
    np.testing.assert_allclose(dX.cpu().numpy(), grads[0].numpy(), rtol=1e-3, atol=1e-4 * sc)
    wk = np.stack([gg.numpy()[:, 0] for gg in grads[1:1 + n]])
    wb = np.stack([gg.numpy()[:, 0] for gg in grads[1 + n:]])
    np.testing.assert_allclose(dK.cpu().numpy(), wk, rtol=1e-3, atol=1e-4 * max(1.0, np.abs(wk).max()))
    np.testing.assert_allclose(dB.cpu().numpy(), wb, rtol=1e-3, atol=1e-4 * max(1.0, np.abs(wb).max()))


# ---------------------------------------------------------------------------------------------
# tensor-core (tcgen05) path
# ---------------------------------------------------------------------------------------------
def _bf16(x):
    return torch.tensor(x).to(torch.bfloat16).to(torch.float32).numpy()


@pytest.mark.parametrize('a_in_tmem', [1, 0])
@pytest.mark.parametrize('n,k', [(128, 64), (32, 16), (64, 32)])
def test_tc_selftest_gemm(nat, a_in_tmem, n, k):
    """One M=128 UMMA tile: validates the instruction / shared-memory descriptors, the TMEM
    operand layout and the accumulator read-back against an exact bf16-input reference."""
    g = np.random.default_rng(20)
    a = g.normal(size=(128, k)).astype(np.float32)
    bm = g.normal(size=(k, n)).astype(np.float32)
    c = torch.zeros(128, n, device='cuda')
    ws = torch.zeros(4 * n * k, dtype=torch.uint8, device='cuda')
    nat.check(nat.lib.dtb_tc_selftest(P(dev(a)), P(dev(bm)), P(c), P(ws), n, k, a_in_tmem, None))
    torch.cuda.synchronize()
    want = _bf16(a).astype(np.float64) @ _bf16(bm).astype(np.float64)
    np.testing.assert_allclose(c.cpu().numpy(), want, rtol=1e-5, atol=1e-4)


TC_CASES = [  # (F, D, sizes, direct, bias, act, B)
    (26, 16, (128, 128, 128), False, False, 1, 37),      # headline shape, ragged tail (37 rows)
    (26, 16, (32, 32, 16), False, False, 1, 64),
    (10, 8, (64, 32), False, True, 1, 50),
    (4, 4, (16, 16), True, False, 1, 70),
    (3, 32, (32, 16), False, True, 0, 9),
    (1, 16, (16,), False, False, 1, 33),
]


@pytest.mark.parametrize('f,d,sizes,direct,use_bias,act,b', TC_CASES)
@pytest.mark.parametrize('precision', [2, 3])
def test_cin_tensor_core_forward(nat, f, d, sizes, direct, use_bias, act, b, precision):
    sizes_c = nat.int_array(sizes)
    n = len(sizes)
    if not nat.lib.dtb_cin_tc_supported(f, d, sizes_c, n, int(direct)):
        pytest.skip('shape not supported by the tensor-core kernels')
    vocab = [9 + i for i in range(f)]
    tabs, flat, offs = make_table(vocab, d, seed=21)
    idx = make_idx(vocab, b, seed=22)
    g = np.random.default_rng(23)
    fns = L.cin_field_nums(f, sizes, direct)
    filt = [(g.normal(size=(f * fns[k], s)) / np.sqrt(f * fns[k])).astype(np.float32) for k, s in enumerate(sizes)]
    bias = [g.normal(size=s).astype(np.float32) * 0.1 for s in sizes] if use_bias else None
    wcat = np.concatenate([x.reshape(-1) for x in filt])
    pw = L.cin_pooled_width(f, dict(cross_layer_size=sizes, direct=direct))
    pooled = torch.full((b, pw), float('nan'), device='cuda')
    ws_bytes = nat.lib.dtb_cin_workspace_bytes(b, f, d, sizes_c, n, int(direct), 1)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device='cuda')
    saved = torch.empty(nat.lib.dtb_cin_saved_bytes(b, f, d, sizes_c, n, int(direct)), dtype=torch.uint8, device='cuda')
    d_b = dev(np.concatenate(bias)) if use_bias else None
    nat.check(nat.lib.dtb_cin_fwd(P(dev(idx)), P(dev(flat)), P(dev(offs)), P(dev(wcat)), P(d_b), P(pooled), P(saved),
                                  P(ws), ws_bytes, b, f, d, sizes_c, n, int(direct), act, precision, None, None))
    torch.cuda.synchronize()
    x = torch.cat(L.embedding_lookup([torch.tensor(t, dtype=torch.float64) for t in tabs], torch.tensor(idx)), dim=1)
    want = _cin_oracle(x, sizes, direct, [torch.tensor(w_, dtype=torch.float64) for w_ in filt],
                       [torch.tensor(b_, dtype=torch.float64) for b_ in bias] if use_bias else None, act).numpy()
    got = pooled.cpu().numpy()
    scale = np.abs(want).max()
    err = np.abs(got - want).max() / scale
    # bf16x3 split: fp32-grade; single bf16 pass: ~2^-8 per operand
    assert err < (2e-5 if precision == 2 else 2e-2), f'max err / scale = {err:.3e}'
    if precision == 2:
        np.testing.assert_allclose(got, want, rtol=1e-3, atol=1e-4 * scale)


def test_cin_fp16_forward_outside_cin_tc2_is_unsupported(nat):
    """Precision 4 forces the single fp16 pass, which only the cin_tc2 kernels run.  On a shape they reject (a
    hidden half of 8 fields: not a multiple of 16) but the bf16x3 kernels take, the forward returns
    DTB_ERR_UNSUPPORTED before it launches anything: workspace and output stay untouched."""
    f, d, sizes, b = 26, 16, (16, 16), 40
    sizes_c, n = nat.int_array(sizes), len(sizes)
    assert nat.lib.dtb_cin_tc_supported(f, d, sizes_c, n, 0)
    vocab = [9 + i for i in range(f)]
    _, flat, offs = make_table(vocab, d, seed=24)
    idx = make_idx(vocab, b, seed=25)
    fns = L.cin_field_nums(f, sizes, False)
    wcat = np.concatenate([np.ones(f * fns[k] * s, np.float32) for k, s in enumerate(sizes)])
    pw = L.cin_pooled_width(f, dict(cross_layer_size=sizes, direct=False))
    pooled = torch.full((b, pw), float('nan'), device='cuda')
    ws_bytes = nat.lib.dtb_cin_workspace_bytes(b, f, d, sizes_c, n, 0, 0)
    ws = torch.full((ws_bytes,), 0x5a, dtype=torch.uint8, device='cuda')
    rc = nat.lib.dtb_cin_fwd(P(dev(idx)), P(dev(flat)), P(dev(offs)), P(dev(wcat)), None, P(pooled), None, P(ws), ws_bytes,
                             b, f, d, sizes_c, n, 0, 1, 4, None, None)
    torch.cuda.synchronize()
    assert rc == -2 and 'cin_tc2' in nat.last_error()                    # DTB_ERR_UNSUPPORTED
    assert bool((ws == 0x5a).all()) and bool(pooled.isnan().all())


def test_cin_tensor_core_full_batch_properties(nat):
    """BASELINE size (65 536 rows, 26x16, CIN 128x128x128): the oracle is too slow, so check
    size-independent properties: duplicated rows give identical outputs, a row permutation permutes
    the output, and a sample of rows matches the exact-fp32 GPU formulation."""
    f, d, sizes, b = 26, 16, (128, 128, 128), 65536
    sizes_c = nat.int_array(sizes)
    vocab = [1000] * f
    tabs, flat, offs = make_table(vocab, d, seed=31)
    idx = make_idx(vocab, b, seed=32)
    idx[1::2] = idx[0::2]                                   # every odd row duplicates the even row before it
    g = np.random.default_rng(33)
    fns = L.cin_field_nums(f, sizes, False)
    wcat = np.concatenate([(g.normal(size=(f * fns[k], s)) / np.sqrt(f * fns[k])).astype(np.float32).reshape(-1)
                           for k, s in enumerate(sizes)])
    d_tab, d_offs, d_w = dev(flat), dev(offs), dev(wcat)

    def run(ix, precision, rows):
        pooled = torch.empty(rows, 256, device='cuda')
        ws_bytes = nat.lib.dtb_cin_workspace_bytes(rows, f, d, sizes_c, 3, 0, 0)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device='cuda')
        nat.check(nat.lib.dtb_cin_fwd(P(dev(ix)), P(d_tab), P(d_offs), P(d_w), None, P(pooled), None, P(ws), ws_bytes,
                                      rows, f, d, sizes_c, 3, 0, 1, precision, None, None))
        return pooled
    out = run(idx, 2, b)
    assert torch.equal(out[0::2], out[1::2])
    perm = np.random.default_rng(34).permutation(b)
    out_p = run(idx[perm], 2, b)
    assert torch.equal(out_p, out[torch.as_tensor(perm, device='cuda')])
    sample = np.arange(0, b, 97)[:512]
    ref = run(idx[sample], 1, len(sample))
    scale = float(ref.abs().max())
    torch.testing.assert_close(out[torch.as_tensor(sample, device='cuda')], ref, rtol=1e-3, atol=1e-4 * scale)


@pytest.mark.parametrize('f,d,sizes,direct,use_bias,act,b', TC_CASES)
def test_cin_tensor_core_backward(nat, f, d, sizes, direct, use_bias, act, b):
    """dgrad + wgrad on tcgen05 (bf16x3) against the oracle's autograd."""
    sizes_c = nat.int_array(sizes)
    n = len(sizes)
    if not nat.lib.dtb_cin_tc_supported(f, d, sizes_c, n, int(direct)):
        pytest.skip('shape not supported by the tensor-core kernels')
    vocab = [9 + i for i in range(f)]
    tabs, flat, offs = make_table(vocab, d, seed=41)
    idx = make_idx(vocab, b, seed=42)
    g = np.random.default_rng(43)
    fns = L.cin_field_nums(f, sizes, direct)
    filt = [(g.normal(size=(f * fns[k], s)) / np.sqrt(f * fns[k])).astype(np.float32) for k, s in enumerate(sizes)]
    bias = [g.normal(size=s).astype(np.float32) * 0.1 for s in sizes] if use_bias else None
    wcat = np.concatenate([x.reshape(-1) for x in filt])
    pw = L.cin_pooled_width(f, dict(cross_layer_size=sizes, direct=direct))
    pooled = torch.empty(b, pw, device='cuda')
    ws_bytes = nat.lib.dtb_cin_workspace_bytes(b, f, d, sizes_c, n, int(direct), 1)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device='cuda')
    saved = torch.empty(nat.lib.dtb_cin_saved_bytes(b, f, d, sizes_c, n, int(direct)), dtype=torch.uint8, device='cuda')
    d_idx, d_tab, d_offs, d_w = dev(idx), dev(flat), dev(offs), dev(wcat)
    d_b = dev(np.concatenate(bias)) if use_bias else None
    dp = g.normal(size=(b, pw)).astype(np.float32)
    d_dp = dev(dp)

    def fwd_bwd():
        gt_ = torch.zeros(flat.shape, device='cuda')
        dw_ = torch.zeros(wcat.shape, device='cuda')
        db_ = torch.zeros(sum(sizes), device='cuda') if use_bias else None
        nat.check(nat.lib.dtb_cin_fwd(P(d_idx), P(d_tab), P(d_offs), P(d_w), P(d_b), P(pooled), P(saved), P(ws),
                                      ws_bytes, b, f, d, sizes_c, n, int(direct), act, 2, None, None))
        nat.check(nat.lib.dtb_cin_bwd(P(d_idx), P(d_tab), P(d_offs), P(d_w), P(d_dp), P(saved), P(gt_), P(dw_), P(db_),
                                      P(ws), ws_bytes, b, f, d, sizes_c, n, int(direct), act, 2, None))
        torch.cuda.synchronize()
        return gt_, dw_, db_

    # (0) default = compact saved activations (relu-mask bits + the operand tiles); bit 17 keeps the fp32 T_k
    #     rows.  Same arithmetic on the same values: only the order of the fp32 atomics may differ.
    gt_c, dw_c, db_c = fwd_bwd()
    nat.lib.dtb_cin_tc_set_variant(1 | (1 << 17))
    try:
        gt, dw, dbias = fwd_bwd()
    finally:
        nat.lib.dtb_cin_tc_set_variant(1)
    for a_, b_, what in ((gt_c, gt, 'embedding grad'), (dw_c, dw, 'filter grad'), (db_c, dbias, 'bias grad')):
        if a_ is not None:
            e = float((a_ - b_).abs().max() / b_.abs().max())
            assert e < 2e-6, f'compact vs full saved activations, {what}: {e:.2e}'
    # (1) same saved activations (=> identical relu masks) through the exact-fp32 backward: the two
    #     backward implementations must agree to bf16x3 precision
    gt2 = torch.zeros(flat.shape, device='cuda')
    dw2 = torch.zeros(wcat.shape, device='cuda')
    db2 = torch.zeros(sum(sizes), device='cuda') if use_bias else None
    nat.lib.dtb_cin_tc_set_variant(1 | (1 << 16) | (1 << 17))
    try:
        nat.check(nat.lib.dtb_cin_bwd(P(d_idx), P(d_tab), P(d_offs), P(d_w), P(d_dp), P(saved), P(gt2), P(dw2), P(db2),
                                      P(ws), ws_bytes, b, f, d, sizes_c, n, int(direct), act, 2, None))
        torch.cuda.synchronize()
    finally:
        nat.lib.dtb_cin_tc_set_variant(1)
    et = float((gt - gt2).abs().max() / gt2.abs().max())
    ew = float((dw - dw2).abs().max() / dw2.abs().max())
    assert et < 5e-5 and ew < 5e-5, f'tensor-core vs fp32 backward: embedding grad {et:.2e}, filter grad {ew:.2e}'
    if use_bias:
        eb = float((dbias - db2).abs().max() / db2.abs().max())
        assert eb < 5e-5, f'bias grad {eb:.2e}'
    # (2) against the oracle's autograd.  A relu unit whose pre-activation is within rounding of zero
    #     may flip between the bf16x3 forward and the float64 oracle, so this bound is looser.
    t64 = [torch.tensor(t, dtype=torch.float64, requires_grad=True) for t in tabs]
    x = torch.cat(L.embedding_lookup(t64, torch.tensor(idx)), dim=1)
    f64 = [torch.tensor(w_, dtype=torch.float64, requires_grad=True) for w_ in filt]
    b64 = [torch.tensor(b_, dtype=torch.float64, requires_grad=True) for b_ in bias] if use_bias else None
    want = _cin_oracle(x, sizes, direct, f64, b64, act)
    loss = (want * torch.tensor(dp, dtype=torch.float64)).sum()
    grads = torch.autograd.grad(loss, t64 + f64 + (b64 or []), allow_unused=True)
    want_t = torch.cat(grads[:f], dim=0).numpy()
    want_w = np.concatenate([gg.numpy().reshape(-1) for gg in grads[f:f + n]])
    et = np.abs(gt.cpu().numpy() - want_t).max() / np.abs(want_t).max()
    ew = np.abs(dw.cpu().numpy() - want_w).max() / np.abs(want_w).max()
    assert et < 1e-2 and ew < 1e-2, f'vs oracle: embedding grad err {et:.2e}, filter grad err {ew:.2e} (relative to max)'


# ---------------------------------------------------------------------------------------------
# PNN products and the AutoInt attention core
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize('f,d,b', [(26, 16, 70), (5, 4, 33), (2, 8, 9), (7, 3, 20), (6, 32, 150), (26, 16, 300), (12, 8, 200)])
@pytest.mark.parametrize('ktype', ['mat', 'vec', 'num'])
def test_pnn_fwd_bwd(nat, f, d, b, ktype):
    vocab = [11 + i for i in range(f)]
    tabs, flat, offs = make_table(vocab, d, seed=51)
    idx = make_idx(vocab, b, seed=52)
    idx[1] = idx[0]
    g = np.random.default_rng(53)
    pairs = f * (f - 1) // 2
    shape = {'mat': (d, pairs, d), 'vec': (pairs, d), 'num': (pairs, 1)}[ktype]
    kern = (g.normal(size=shape) / np.sqrt(d)).astype(np.float32)
    kt = {'mat': 0, 'vec': 1, 'num': 2}[ktype]
    d_idx, d_tab, d_offs, d_k = dev(idx), dev(flat), dev(offs), dev(kern)
    ip = torch.empty(b, pairs, device='cuda')
    op = torch.empty(b, pairs, device='cuda')
    nat.check(nat.lib.dtb_pnn_fwd(P(d_idx), P(d_tab), P(d_offs), P(d_k), P(ip), P(op), b, f, d, kt, None, None))
    t64 = [torch.tensor(t, dtype=torch.float64, requires_grad=True) for t in tabs]
    emb = L.embedding_lookup(t64, torch.tensor(idx))
    k64 = torch.tensor(kern, dtype=torch.float64, requires_grad=True)
    want_ip = L.inner_product(emb)
    want_op = L.outer_product(emb, k64, ktype)
    np.testing.assert_allclose(ip.cpu().numpy(), want_ip.detach().numpy(), rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(op.cpu().numpy(), want_op.detach().numpy(), rtol=1e-4, atol=1e-5)
    g_ip = g.normal(size=(b, pairs)).astype(np.float32)
    g_op = g.normal(size=(b, pairs)).astype(np.float32)
    gt = torch.zeros(flat.shape, device='cuda')
    dk = torch.zeros(kern.shape, device='cuda')
    nat.check(nat.lib.dtb_pnn_bwd(P(d_idx), P(d_tab), P(d_offs), P(d_k), P(dev(g_ip)), P(dev(g_op)), P(gt), P(dk), b, f, d,
                                  kt, None))
    loss = (want_ip * torch.tensor(g_ip, dtype=torch.float64)).sum() + (want_op * torch.tensor(g_op, dtype=torch.float64)).sum()
    grads = torch.autograd.grad(loss, t64 + [k64])
    want_t = torch.cat(grads[:-1], dim=0).numpy()
    np.testing.assert_allclose(gt.cpu().numpy(), want_t, rtol=1e-3, atol=1e-4 * np.abs(want_t).max())
    np.testing.assert_allclose(dk.cpu().numpy(), grads[-1].numpy(), rtol=1e-3, atol=1e-4 * np.abs(grads[-1].numpy()).max())


@pytest.mark.parametrize('f,d,h,b,act', [(26, 16, 16, 70, 'relu'), (5, 4, 5, 33, 'linear'), (3, 8, 32, 200, 'relu'),
                                         (7, 32, 8, 20, 'relu'), (2, 16, 4, 9, 'relu'), (12, 8, 16, 300, 'relu')])
def test_afm_fwd_bwd(nat, f, d, h, b, act):
    """AFM attention pooling (layers.py:790-804) and its gradients against the fp64 oracle's autograd."""
    vocab = [11 + i for i in range(f)]
    tabs, flat, offs = make_table(vocab, d, seed=61)
    idx = make_idx(vocab, b, seed=62)
    idx[1] = idx[0]
    g = np.random.default_rng(63)
    wa = (g.normal(size=(d, h)) / np.sqrt(d)).astype(np.float32) * 3
    ba = (g.normal(size=(h,)) * 0.1).astype(np.float32)
    ph = g.normal(size=(h, 1)).astype(np.float32)
    act_code = {'linear': 0, 'relu': 1}[act]
    d_idx, d_tab, d_offs, d_wa, d_ba, d_ph = dev(idx), dev(flat), dev(offs), dev(wa), dev(ba), dev(ph)
    pooled = torch.empty(b, d, device='cuda')
    nat.check(nat.lib.dtb_afm_fwd(P(d_idx), P(d_tab), P(d_offs), P(d_wa), P(d_ba), P(d_ph), P(pooled), b, f, d, h, act_code, None,
                                  None))
    t64 = [torch.tensor(t, dtype=torch.float64, requires_grad=True) for t in tabs]
    w64 = [torch.tensor(a, dtype=torch.float64, requires_grad=True) for a in (wa, ba, ph)]
    emb = L.embedding_lookup(t64, torch.tensor(idx))
    want = L.afm_pooled(emb, w64[0], w64[1], w64[2], act)
    np.testing.assert_allclose(pooled.cpu().numpy(), want.detach().numpy(), rtol=1e-4, atol=1e-5 * float(want.abs().max()))
    gp = g.normal(size=(b, d)).astype(np.float32)
    gt = torch.zeros(flat.shape, device='cuda')
    dwa, dba, dph = torch.zeros(d, h, device='cuda'), torch.zeros(h, device='cuda'), torch.zeros(h, 1, device='cuda')
    nb = nat.lib.dtb_afm_workspace_bytes(b, f, d, h)
    ws = torch.empty(nb, dtype=torch.uint8, device='cuda')
    nat.check(nat.lib.dtb_afm_bwd(P(d_idx), P(d_tab), P(d_offs), P(d_wa), P(d_ba), P(d_ph), P(dev(gp)), P(gt), P(dwa), P(dba), P(dph),
                                  P(ws), nb, b, f, d, h, act_code, None))
    grads = torch.autograd.grad((want * torch.tensor(gp, dtype=torch.float64)).sum(), t64 + w64)
    want_t = torch.cat(grads[:f], dim=0).numpy()
    scale = 1e-2 * float(np.abs(grads[f].numpy()).max())
    for name, got, ref in (('table', gt, want_t), ('att_kernel', dwa, grads[f].numpy()), ('att_bias', dba, grads[f + 1].numpy()),
                           ('projection_h', dph, grads[f + 2].numpy())):
        # (with a linear attention the bias gradient is exactly zero -- the softmax ignores a common shift -- so the floor
        # of the tolerance is the scale of the kernel gradient, not of the reference value)
        np.testing.assert_allclose(got.cpu().numpy(), ref, rtol=2e-3, atol=2e-4 * max(np.abs(ref).max(), scale), err_msg=name)


@pytest.mark.parametrize('f,d,b', [(26, 16, 150), (5, 4, 33), (2, 8, 9), (7, 32, 130), (12, 8, 300)])
@pytest.mark.parametrize('bt', ['field_all', 'field_each', 'field_interaction'])
def test_bilinear_fwd_bwd(nat, f, d, b, bt):
    """BilinearInteraction (layers.py:358-372) on a dense block and its gradients against the fp64 oracle's autograd."""
    g = np.random.default_rng(71)
    pairs = f * (f - 1) // 2
    n_w = {'field_all': 1, 'field_each': f - 1, 'field_interaction': pairs}[bt]
    code = {'field_all': 0, 'field_each': 1, 'field_interaction': 2}[bt]
    x = g.normal(size=(b, f, d)).astype(np.float32)
    w = (g.normal(size=(n_w, d, d)) / np.sqrt(d)).astype(np.float32)
    d_x, d_w = dev(x), dev(w)
    out = torch.empty(b, pairs, d, device='cuda')
    nat.check(nat.lib.dtb_bilinear_fwd(P(d_x), P(d_w), P(out), b, f, d, code, None))
    x64 = torch.tensor(x, dtype=torch.float64, requires_grad=True)
    w64 = torch.tensor(w, dtype=torch.float64, requires_grad=True)
    want = L.bilinear_interaction(x64, list(w64), bt)
    np.testing.assert_allclose(out.cpu().numpy(), want.detach().numpy(), rtol=1e-4, atol=1e-5 * float(want.abs().max()))
    go = g.normal(size=(b, pairs, d)).astype(np.float32)
    dx, dw = torch.empty(b, f, d, device='cuda'), torch.zeros(n_w, d, d, device='cuda')
    nat.check(nat.lib.dtb_bilinear_bwd(P(d_x), P(d_w), P(dev(go)), P(dx), P(dw), b, f, d, code, None))
    gx, gw = torch.autograd.grad((want * torch.tensor(go, dtype=torch.float64)).sum(), [x64, w64])
    np.testing.assert_allclose(dx.cpu().numpy(), gx.numpy(), rtol=1e-3, atol=1e-4 * float(gx.abs().max()))
    np.testing.assert_allclose(dw.cpu().numpy(), gw.numpy(), rtol=1e-3, atol=1e-4 * float(gw.abs().max()))


@pytest.mark.parametrize('task,cols,gamma,alpha', [(0, 1, 2.0, 0.25), (0, 3, 1.5, 0.6), (0, 1, 0.0, 0.5), (2, 4, 2.0, 0.25), (2, 3, 0.5, 1.0)])
def test_focal_loss_fwd_bwd(nat, task, cols, gamma, alpha):
    """Binary / categorical focal loss (layers.py:983-1083) on the task_output pre-activation against the oracle's autograd."""
    g = np.random.default_rng(91)
    rows = 257
    z = (g.normal(size=(rows, cols)) * 3).astype(np.float32)
    z[0, 0], z[1, 0] = 30.0, -30.0                                  # saturated probabilities: the clip turns the gradient off
    if task == 0:
        y = (g.random((rows, cols)) < 0.4).astype(np.float32)
    else:
        y = np.eye(cols, dtype=np.float32)[g.integers(0, cols, size=rows)]
    prob, dz = torch.empty(rows, cols, device='cuda'), torch.empty(rows, cols, device='cuda')
    acc = torch.zeros(1, dtype=torch.float64, device='cuda')
    nat.check(nat.lib.dtb_focal_loss_fwd_bwd(P(dev(z)), P(dev(y)), P(prob), P(dz), P(acc), rows, cols, task, gamma, alpha, None))
    z64 = torch.tensor(z, dtype=torch.float64, requires_grad=True)
    y64 = torch.tensor(y, dtype=torch.float64)
    if task == 0:
        p64 = torch.sigmoid(z64)
        loss = L.binary_focal_loss(y64, p64, gamma, alpha)
    else:
        p64 = torch.softmax(z64, dim=-1)
        loss = L.categorical_focal_loss(y64, p64, gamma, alpha).mean()
    (gz,) = torch.autograd.grad(loss, [z64])
    np.testing.assert_allclose(prob.cpu().numpy(), p64.detach().numpy(), rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(float(acc.item()) / rows, float(loss), rtol=2e-5)
    # fp32 probabilities saturate (1 - p = 0 or p clipped) where float64 does not: compare where the fp32 probability is interior
    interior = (prob.cpu().numpy() > 1e-6) & (prob.cpu().numpy() < 1 - 1e-6)
    if task == 2:
        interior = np.repeat(interior.all(axis=1, keepdims=True), cols, axis=1)
    np.testing.assert_allclose(dz.cpu().numpy()[interior], gz.numpy()[interior], rtol=2e-3, atol=1e-6 / rows)


@pytest.mark.parametrize('b,h,w,cin,cout,kh,pool,act', [(9, 26, 16, 1, 14, 7, 2, 'tanh'), (5, 13, 16, 14, 16, 7, 2, 'tanh'),
                                                        (7, 7, 4, 3, 4, 4, 3, 'relu'), (33, 5, 8, 32, 32, 8, 5, 'linear'),
                                                        (300, 3, 4, 2, 5, 1, 1, 'tanh')])
def test_fgcnn_conv_and_pool_fwd_bwd(nat, b, h, w, cin, cout, kh, pool, act):
    """FGCNN's convolution and max pooling along the field axis (layers.py:204-214) against the fp64 oracle's autograd."""
    g = np.random.default_rng(81)
    x = g.normal(size=(b, h, w, cin)).astype(np.float32)
    k = (g.normal(size=(kh, 1, cin, cout)) / np.sqrt(kh * cin)).astype(np.float32)
    bias = (g.normal(size=(cout,)) * 0.1).astype(np.float32)
    code = {'linear': 0, 'relu': 1, 'tanh': 2}[act]
    d_x, d_k, d_b = dev(x), dev(k), dev(bias)
    y = torch.empty(b, h, w, cout, device='cuda')
    nat.check(nat.lib.dtb_conv_fields_fwd(P(d_x), P(d_k), P(d_b), P(y), b, h, w, cin, cout, kh, code, None))
    x64 = torch.tensor(x, dtype=torch.float64, requires_grad=True)
    k64 = torch.tensor(k, dtype=torch.float64, requires_grad=True)
    b64 = torch.tensor(bias, dtype=torch.float64, requires_grad=True)
    want = L.conv_fields(x64, k64, b64, act)
    np.testing.assert_allclose(y.cpu().numpy(), want.detach().numpy(), rtol=1e-4, atol=1e-5)
    ho = -(-h // pool)
    pooled = torch.empty(b, ho, w, cout, device='cuda')
    nat.check(nat.lib.dtb_maxpool_fields_fwd(P(y), P(pooled), b, h, w * cout, pool, None))
    want_p = L.maxpool_fields(want, pool)
    np.testing.assert_allclose(pooled.cpu().numpy(), want_p.detach().numpy(), rtol=1e-4, atol=1e-5)
    gp = g.normal(size=(b, ho, w, cout)).astype(np.float32)
    dy = torch.empty_like(y)
    nat.check(nat.lib.dtb_maxpool_fields_bwd(P(y), P(dev(gp)), P(dy), b, h, w * cout, pool, None))
    dx, dk, db = torch.empty_like(d_x), torch.zeros_like(d_k), torch.zeros_like(d_b)
    nat.check(nat.lib.dtb_conv_fields_bwd(P(d_x), P(d_k), P(y), P(dy), P(dx), P(dk), P(db), b, h, w, cin, cout, kh, code, None))
    gy, = torch.autograd.grad((want_p * torch.tensor(gp, dtype=torch.float64)).sum(), [want], retain_graph=True)
    gx, gk, gb = torch.autograd.grad((want_p * torch.tensor(gp, dtype=torch.float64)).sum(), [x64, k64, b64])
    np.testing.assert_allclose(dy.cpu().numpy(), gy.numpy(), rtol=1e-4, atol=1e-6)
    for name, got, ref in (('dx', dx, gx), ('dk', dk, gk), ('db', db, gb)):
        np.testing.assert_allclose(got.cpu().numpy(), ref.numpy(), rtol=2e-3, atol=2e-4 * float(ref.abs().max()), err_msg=name)


def test_dense_tanh_activation(nat):
    """DTB_ACT_TANH in the Dense epilogues (wide: tcgen05 path, narrow: row-dot path) and its backward."""
    g = np.random.default_rng(82)
    for rows, i, o in ((300, 36, 40), (200, 48, 5)):
        x = g.normal(size=(rows, i)).astype(np.float32)
        w = (g.normal(size=(i, o)) / np.sqrt(i)).astype(np.float32)
        bias = (g.normal(size=(o,)) * 0.1).astype(np.float32)
        d_x, d_w, d_b = dev(x), dev(w), dev(bias)
        y = torch.empty(rows, o, device='cuda')
        nb = nat.lib.dtb_dense_workspace_bytes(i, o)
        ws = torch.empty(max(nb, 16), dtype=torch.uint8, device='cuda')
        nat.check(nat.lib.dtb_dense_fwd(P(d_x), P(d_w), P(d_b), P(y), P(ws), nb, rows, i, o, 2, None))
        x64, w64, b64 = (torch.tensor(a, dtype=torch.float64, requires_grad=True) for a in (x, w, bias))
        want = torch.tanh(x64 @ w64 + b64)
        np.testing.assert_allclose(y.cpu().numpy(), want.detach().numpy(), rtol=1e-4, atol=2e-5)
        gy = g.normal(size=(rows, o)).astype(np.float32)
        dyv, dx, dw, db = dev(gy), torch.empty_like(d_x), torch.zeros_like(d_w), torch.zeros_like(d_b)
        y_ref = torch.tensor(want.detach().numpy().astype(np.float32)).cuda()        # the oracle's outputs: same tanh' on both sides
        nat.check(nat.lib.dtb_dense_bwd(P(d_x), P(d_w), P(y_ref), P(dyv), P(dx), P(dw), P(db), P(ws), nb, rows, i, o, 2, None))
        gx, gw, gb = torch.autograd.grad((want * torch.tensor(gy, dtype=torch.float64)).sum(), [x64, w64, b64])
        for name, got, ref in (('dx', dx, gx), ('dw', dw, gw), ('db', db, gb)):
            np.testing.assert_allclose(got.cpu().numpy(), ref.numpy(), rtol=2e-3, atol=2e-4 * float(ref.abs().max()), err_msg=name)


@pytest.mark.parametrize('op', ['mean', 'max'])
def test_senet_pool_and_scale(nat, op):
    """SENET squeeze / re-weighting kernels (layers.py:291-303) against torch autograd on the same arithmetic."""
    g = np.random.default_rng(72)
    b, f, d = 37, 7, 8
    x = g.normal(size=(b, f, d)).astype(np.float32)
    x[3, 2, 1] = x[3, 2, 5] = 9.0                                  # a tie of the maximum: the gradient is shared
    a = np.abs(g.normal(size=(b, f))).astype(np.float32)
    d_x, d_a = dev(x), dev(a)
    z, v = torch.empty(b, f, device='cuda'), torch.empty(b, f, d, device='cuda')
    code = 1 if op == 'max' else 0
    nat.check(nat.lib.dtb_senet_pool_fwd(P(d_x), P(z), b, f, d, code, None))
    nat.check(nat.lib.dtb_senet_scale_fwd(P(d_x), P(d_a), P(v), b, f, d, None))
    x64 = torch.tensor(x, dtype=torch.float64, requires_grad=True)
    a64 = torch.tensor(a, dtype=torch.float64, requires_grad=True)
    want_z = x64.amax(dim=-1) if op == 'max' else x64.mean(dim=-1)
    want_v = x64 * a64.unsqueeze(2)
    np.testing.assert_allclose(z.cpu().numpy(), want_z.detach().numpy(), rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(v.cpu().numpy(), want_v.detach().numpy(), rtol=1e-6, atol=1e-7)
    gz, gv = g.normal(size=(b, f)).astype(np.float32), g.normal(size=(b, f, d)).astype(np.float32)
    dxz, dxv, da = torch.empty(b, f, d, device='cuda'), torch.empty(b, f, d, device='cuda'), torch.empty(b, f, device='cuda')
    nat.check(nat.lib.dtb_senet_pool_bwd(P(d_x), P(z), P(dev(gz)), P(dxz), b, f, d, code, None))
    nat.check(nat.lib.dtb_senet_scale_bwd(P(d_x), P(d_a), P(dev(gv)), P(dxv), P(da), b, f, d, None))
    (wz,) = torch.autograd.grad((want_z * torch.tensor(gz, dtype=torch.float64)).sum(), [x64])
    wv, wa = torch.autograd.grad((want_v * torch.tensor(gv, dtype=torch.float64)).sum(), [x64, a64])
    np.testing.assert_allclose(dxz.cpu().numpy(), wz.numpy(), rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(dxv.cpu().numpy(), wv.numpy(), rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(da.cpu().numpy(), wa.numpy(), rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize('b,f,d,heads,res', [(40, 26, 32, 4, True), (17, 5, 4, 1, True), (9, 7, 16, 2, False), (3, 1, 8, 8, True),
                                               (1001, 26, 16, 1, True), (131, 26, 32, 4, False), (70, 3, 64, 1, True)])
def test_attention_core_fwd_bwd(nat, b, f, d, heads, res):
    g = np.random.default_rng(54)
    qkvr = np.maximum(g.normal(size=(b, f, 4 * d)), 0).astype(np.float32)       # relu outputs
    y = torch.empty(b, f, d, device='cuda')
    d_in = dev(qkvr)
    nat.check(nat.lib.dtb_attention_core_fwd(P(d_in), P(y), b, f, d, heads, int(res), None))
    x64 = torch.tensor(qkvr, dtype=torch.float64, requires_grad=True)
    q, k, v, r = torch.split(x64, d, dim=-1)
    q_ = torch.cat(torch.chunk(q, heads, dim=2), dim=0)
    k_ = torch.cat(torch.chunk(k, heads, dim=2), dim=0)
    v_ = torch.cat(torch.chunk(v, heads, dim=2), dim=0)
    w = torch.softmax(q_ @ k_.transpose(1, 2) / (k_.shape[-1] ** 0.5), dim=-1)
    out = torch.cat(torch.chunk(w @ v_, heads, dim=0), dim=2)
    if res:
        out = out + r
    want = torch.relu(out)
    np.testing.assert_allclose(y.cpu().numpy(), want.detach().numpy(), rtol=1e-4, atol=1e-5)
    dy = g.normal(size=(b, f, d)).astype(np.float32)
    dq = torch.empty(b, f, 4 * d, device='cuda')
    nat.check(nat.lib.dtb_attention_core_bwd(P(d_in), P(y), P(dev(dy)), P(dq), b, f, d, heads, int(res), 0, None))
    (gx,) = torch.autograd.grad((want * torch.tensor(dy, dtype=torch.float64)).sum(), [x64])
    np.testing.assert_allclose(dq.cpu().numpy(), gx.numpy(), rtol=1e-3, atol=1e-4 * max(1.0, float(gx.abs().max())))
    # mask_relu_inputs: the same gradient, zeroed where the (relu-output) input is zero
    dqm = torch.empty(b, f, 4 * d, device='cuda')
    nat.check(nat.lib.dtb_attention_core_bwd(P(d_in), P(y), P(dev(dy)), P(dqm), b, f, d, heads, int(res), 1, None))
    assert torch.equal(dqm, dq * (d_in.view(b, f, 4 * d) > 0))
