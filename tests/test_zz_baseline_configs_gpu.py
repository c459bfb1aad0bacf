"""BASELINE.json configs [1], [3], [4] at their FULL shapes (Criteo: 26 sparse x vocab 1M + 13 dense), as parity-test
cases: the oracle cannot hold 1.66 GB tables comfortably, so each case checks size-independent properties on the
whole batch and compares a sample of rows against the CPU oracle run on a compacted copy of the weights
(only the embedding rows those sample rows reference).
"""
import numpy as np
import pytest
import torch

from oracle import model_ref as M

pytestmark = [pytest.mark.gpu]

F, C, V = 26, 13, 1_000_000

CASES = {
    # config [1]: DeepFM, embed_dim 16, bs 8192
    'deepfm_bs8192': dict(nets=['linear', 'fm_nets', 'dnn_nets'], dim=16, batch=8192, kw={}),
    # config [3]: DCN CrossNet depth 6 stacked with AutoInt 4-head d=32, bs 65536
    'dcn6_autoint4x32_bs65536': dict(nets=['dcn_nets', 'autoint_nets'], dim=32, batch=65536,
                                     kw=dict(cross_params={'num_cross_layer': 6},
                                             autoint_params={'num_attention': 3, 'num_heads': 4, 'dropout_rate': 0,
                                                             'use_residual': True})),
    # config [4]: the five-net mix; 131072 global rows over 8 GPUs = 16384 per GPU
    'five_nets_bs16384': dict(nets=['fm_nets', 'cin_nets', 'cross_nets', 'autoint_nets', 'pnn_nets'], dim=16, batch=16384,
                              kw=dict(cin_params={'cross_layer_size': (128, 128, 128), 'activation': 'relu',
                                                  'use_residual': False, 'use_bias': False, 'direct': False,
                                                  'reduce_D': False})),
}


def _build(nets, dim, kw):
    from deeptables_b200 import deeptable
    from deeptables_b200.deepmodel import DeepModel
    from deeptables_b200.metainfo import CategoricalColumn, ContinuousColumn
    conf = deeptable.ModelConfig(nets=nets, embeddings_output_dim=dim, embedding_dropout=0, metrics=['AUC'], **kw)
    cats = [CategoricalColumn(f'C{i + 1}', V, dim) for i in range(F)]
    conts = [ContinuousColumn('input_continuous_all', [f'I{i + 1}' for i in range(C)])]
    model = DeepModel('binary', 2, conf, cats, conts, seed=21)
    model._build_model()
    return model, conf


@pytest.mark.parametrize('case', sorted(CASES))
def test_baseline_config_full_shape(case):
    spec = CASES[case]
    model, conf = _build(spec['nets'], spec['dim'], spec['kw'])
    b, dim = spec['batch'], spec['dim']
    g = torch.Generator().manual_seed(5)
    idx = torch.randint(0, V, (b, F), generator=g, dtype=torch.int32)
    cont = torch.randn(b, C, generator=g)
    half = b // 2
    idx[half:] = idx[:half]                                   # duplicated rows
    cont[half:] = cont[:half]
    d_idx, d_cont = idx.cuda(), cont.cuda()
    out = model.predict_step(d_idx, d_cont)
    assert out.shape == (b, 1) and bool(torch.isfinite(out).all())
    # (1) duplicated rows give identical outputs (no cross-row coupling in inference)
    torch.testing.assert_close(out[:half], out[half:], rtol=1e-6, atol=1e-7)
    # (2) a row permutation permutes the output
    perm = torch.randperm(b, generator=g)
    out_p = model.predict_step(d_idx[perm.cuda()], d_cont[perm.cuda()])
    torch.testing.assert_close(out_p, out[perm.cuda()], rtol=1e-5, atol=1e-6)
    # (3) a sample of rows against the oracle, on weights compacted to the rows the sample references
    sample = torch.arange(0, half, max(1, half // 48))[:48]
    s_idx = idx[sample]
    state = {}
    sd = model.state_dict()
    for i in range(F):
        rows = s_idx[:, i].long().cuda()
        state[f'emb_categorical_vars_all/embeddings_{i}'] = sd[f'emb_categorical_vars_all/embeddings_{i}'][rows].cpu()
    for k, v in sd.items():
        if not k.startswith('emb_categorical_vars_all/'):
            state[k] = v.detach().cpu().clone()
    local_ids = torch.arange(len(sample), dtype=torch.int64).unsqueeze(1).repeat(1, F)   # row r of every compact table
    want, _ = M.forward(state, conf, local_ids, cont[sample], F, False)
    torch.testing.assert_close(out[sample.cuda()].cpu(), want, rtol=1e-3, atol=1e-5)      # north_star: 1e-3 relative fp32
    # (4) a few optimiser steps at the full shape stay finite and reduce the loss on a fixed batch
    y = (torch.rand(b, generator=g) < 0.25).float().numpy()
    losses = [model.train_on_batch(idx.numpy(), cont.numpy(), y) for _ in range(4)]
    assert np.isfinite(losses).all() and losses[-1] < losses[0]
    model.release()


# ---------------------------------------------------------------------------------------------------------------
# DTB_CIN_TC_F16X1 (precision code 4): single tensor pass on power-of-two-scaled fp16 operands
# ---------------------------------------------------------------------------------------------------------------
F16_CASES = [  # (F, sizes, direct, bias, act, B, D): the two-threads-per-GEMM-row kernels of cin_tc2.cu
    (26, (128, 128, 128), False, False, 1, 37, 16),
    (26, (32, 32, 16), False, True, 1, 64, 16),
    (10, (64, 32), True, True, 1, 50, 16),
    (3, (32, 16), False, False, 0, 9, 16),
    (26, (128, 128), False, False, 1, 21, 32),
    (40, (96, 64, 48), False, True, 1, 300, 16),      # F > 32: layer 0 is a 64-wide chunk too; ragged pooled split
]


@pytest.mark.parametrize('f,sizes,direct,use_bias,act,b,d', F16_CASES)
def test_cin_fp16_single_pass_forward_is_inside_the_parity_bar(f, sizes, direct, use_bias, act, b, d):
    """tools/cin_precision_study.py predicts max |err| of 2-6e-4 of the output scale for this scheme; the parity
    bar is rtol 1e-3 (+ atol 1e-4 of the scale).  Also checks that a backward (bf16x3 kernels) runs on the
    activations this forward saved."""
    import ctypes
    from deeptables_b200 import _native as nat
    from oracle import layers_ref as L
    P = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())     # noqa: E731
    g = np.random.default_rng(61)
    vocab = [9 + i for i in range(f)]
    offs = np.concatenate([[0], np.cumsum(vocab)]).astype(np.int64)
    table = ((g.random((int(offs[-1]), d)) - 0.5) * 0.1).astype(np.float32)
    idx = np.stack([g.integers(0, v, size=b) for v in vocab], axis=1).astype(np.int32)
    fns = L.cin_field_nums(f, sizes, direct)
    filt = [(g.normal(size=(f * fns[k], s)) / np.sqrt(f * fns[k])).astype(np.float32) for k, s in enumerate(sizes)]
    bias = [g.normal(size=s).astype(np.float32) * 0.1 for s in sizes] if use_bias else None
    sizes_c, n = nat.int_array(sizes), len(sizes)
    if not nat.lib.dtb_cin_tc_supported(f, d, sizes_c, n, int(direct)):
        pytest.skip('shape not supported by the tensor-core kernels')
    params = dict(cross_layer_size=sizes, direct=direct, use_bias=use_bias, activation='relu' if act else 'linear')
    pw = L.cin_pooled_width(f, params)
    dev = lambda a: torch.tensor(a).cuda()                                   # noqa: E731
    d_idx, d_tab, d_offs = dev(idx), dev(table), dev(offs)
    d_w = dev(np.concatenate([x.reshape(-1) for x in filt]))
    d_b = dev(np.concatenate(bias)) if use_bias else None
    pooled = torch.empty(b, pw, device='cuda')
    ws_bytes = nat.lib.dtb_cin_workspace_bytes(b, f, d, sizes_c, n, int(direct), 1)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device='cuda')
    saved = torch.empty(nat.lib.dtb_cin_saved_bytes(b, f, d, sizes_c, n, int(direct)), dtype=torch.uint8, device='cuda')
    nat.check(nat.lib.dtb_cin_fwd(P(d_idx), P(d_tab), P(d_offs), P(d_w), P(d_b), P(pooled), P(saved), P(ws), ws_bytes,
                                  b, f, d, sizes_c, n, int(direct), act, 4, None, None), 'cin_fwd fp16x1')
    torch.cuda.synchronize()
    # float64 reference of the pooled feature maps (the oracle's CIN up to the sum over D: identity output kernels)
    t64 = torch.tensor(table, dtype=torch.float64)
    x = torch.stack([t64[offs[i] + torch.tensor(idx[:, i].astype(np.int64))] for i in range(f)], dim=1)
    outs = []
    for col in range(pw):
        w = {f'f_{k}': torch.tensor(filt[k], dtype=torch.float64).unsqueeze(0) for k in range(n)}
        if use_bias:
            w.update({f'bias{k}': torch.tensor(bias[k], dtype=torch.float64) for k in range(n)})
        kern = torch.zeros(pw, 1, dtype=torch.float64)
        kern[col, 0] = 1.0
        w['exFM_out/kernel'], w['exFM_out/bias'] = kern, torch.zeros(1, dtype=torch.float64)
        outs.append(L.cin(x, params, w))
    want = torch.cat(outs, dim=1).numpy()
    got = pooled.cpu().double().numpy()
    scale = np.abs(want).max()
    # one fp16 pass rounds each operand to 2^-11: the error of an output is ~3e-4 of the magnitude of its terms, NOT of
    # the output itself -- entries that are small through cancellation (tiny F, linear activation) carry the same
    # absolute error as their neighbours.  Bar: 1e-3 of the output scale everywhere, and 1e-3 relative wherever the
    # entry is not itself below 1 % of the scale.
    err = np.abs(got - want)
    assert err.max() / scale < 1e-3, f'max error {err.max() / scale:.2e} of the output scale'
    big = np.abs(want) > 1e-2 * scale
    print(f'fp16x1 F={f} sizes={sizes}: max err / scale {err.max() / scale:.2e}, '
          f'max rel err on entries > 1% of scale {(err[big] / np.abs(want[big])).max():.2e}')
    # elementwise: 1e-3 relative plus 1e-4 of the scale -- except for tiny reductions (F*H < 64 terms per output) where
    # the rounding errors of the few terms do not average out and the norm-wise bound above is all one fp16 pass gives
    if f * min(L.cin_field_nums(f, sizes, direct)) >= 64:
        bad = err > 1e-3 * np.abs(want) + 1e-4 * scale + 4e-4 * scale * (~big)
        assert not bad.any(), f'{int(bad.sum())} entries outside the bar, worst {err[bad].max() / scale:.2e} of the scale'
    # backward: the fp16 single-pass kernels (cin_tc2 dgrad + fp16 wgrad) against the bf16x3 kernels ON THE SAME saved
    # activations (the fp16 forward's: a different forward flips relu-mask bits of near-zero outputs, which moves single
    # gradient rows by percents and says nothing about the backward arithmetic)
    d_dp = torch.randn(b, pw, device='cuda', generator=torch.Generator(device='cuda').manual_seed(5))

    def backward(prec_b):
        gt = torch.zeros(table.shape, device='cuda')
        dw = torch.zeros_like(d_w)
        db = torch.zeros(sum(sizes), device='cuda') if use_bias else None
        nat.check(nat.lib.dtb_cin_bwd(P(d_idx), P(d_tab), P(d_offs), P(d_w), P(d_dp), P(saved), P(gt), P(dw), P(db), P(ws),
                                      ws_bytes, b, f, d, sizes_c, n, int(direct), act, prec_b, None), 'cin_bwd')
        torch.cuda.synchronize()
        return gt, dw, db

    ref = backward(2)           # bf16x3 explicitly: 0 = auto resolves to the fp16 kernels where they apply
    assert all(bool(torch.isfinite(t_).all()) for t_ in ref if t_ is not None) and float(ref[1].abs().max()) > 0
    got_g = backward(4)
    for name, r_, g_ in zip(('embedding', 'filter', 'bias'), ref, got_g):
        if r_ is None:
            continue
        assert bool(torch.isfinite(g_).all())
        rel = float((r_ - g_).abs().max() / r_.abs().max())
        print(f'fp16x1 backward, {name} gradient vs bf16x3 on the same activations: max err / max {rel:.2e}')
        assert rel < 2e-3, f'{name} gradient off by {rel:.2e} of its maximum'
