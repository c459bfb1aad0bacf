"""CPU-side tests: the C-ABI library loads and exports every declared symbol; host-side logic
(config, registry, column metadata, preprocessor) behaves like the reference's."""
import inspect
import os

import numpy as np
import pandas as pd
import pytest


def test_library_exports_every_declared_symbol():
    from deeptables_b200 import _native
    declared = _native.declared_symbols()
    assert len(declared) >= 25
    for sym in declared:
        assert hasattr(_native.lib, sym), f'{sym} declared in include/deeptables_b200.h but not exported'
        assert sym in _native._SIGNATURES, f'{sym} has no ctypes signature'
    assert _native.lib.dtb_version() >= 100


def test_graft_build_is_idempotent():
    import __graft_entry__ as g
    path = g.build()
    assert os.path.exists(path)


def test_model_config_defaults_match_reference():
    from deeptables_b200 import deeptable
    c = deeptable.ModelConfig()
    # reference deeptables/models/config.py:59-136
    assert c.name == 'conf-1' and c.nets == ['dnn_nets'] and c.metrics == ['accuracy']
    assert c.embeddings_output_dim == 4 and c.embedding_dropout == 0.3 and c.dense_dropout == 0
    assert c.stacking_op == 'add' and c.output_use_bias is True and c.optimizer == 'auto' and c.loss == 'auto'
    assert c.dnn_params == {'hidden_units': ((128, 0, False), (64, 0, False)), 'activation': 'relu'}
    assert c.cross_params == {'num_cross_layer': 4}
    assert c.cin_params['cross_layer_size'] == (128, 128) and c.cin_params['direct'] is False
    assert c.autoint_params == {'num_attention': 3, 'num_heads': 1, 'dropout_rate': 0, 'use_residual': True}
    assert c.earlystopping_patience == 1 and c.earlystopping_mode == 'auto'
    assert len(c._fields) == 45
    assert c.first_metric_name == 'accuracy'
    # positional order is the reference's
    assert c._fields[:5] == ('name', 'nets', 'categorical_columns', 'exclude_columns', 'task')
    with pytest.raises(TypeError):
        deeptable.ModelConfig(not_a_field=1)
    with pytest.raises(ValueError):
        deeptable.ModelConfig(var_len_categorical_columns=[('a', '|')])
    # defaults are not shared between instances
    c.dnn_params['activation'] = 'x'
    assert deeptable.ModelConfig().dnn_params['activation'] == 'relu'


def test_nets_registry_names_presets_and_signature():
    from deeptables_b200 import deepnets
    assert deepnets.xDeepFM == ['linear', 'cin_nets', 'dnn_nets'] and deepnets.DeepFM == ['linear', 'fm_nets', 'dnn_nets']
    assert deepnets.DCN == ['dcn_nets'] and deepnets.PNN == ['pnn_nets'] and deepnets.AutoInt == ['autoint_nets']
    names = ['linear', 'cin_nets', 'fm_nets', 'afm_nets', 'opnn_nets', 'ipnn_nets', 'pnn_nets', 'dnn_nets', 'cross_nets',
             'cross_dnn_nets', 'dcn_nets', 'autoint_nets', 'fg_nets', 'fgcnn_cin_nets', 'fgcnn_fm_nets',
             'fgcnn_ipnn_nets', 'fgcnn_dnn_nets', 'fibi_nets', 'fibi_dnn_nets']
    sig = inspect.signature(deepnets.linear)
    assert list(sig.parameters) == ['embeddings', 'flatten_emb_layer', 'dense_layer', 'concat_emb_dense', 'config',
                                    'model_desc']
    for n in names:
        fn = deepnets.get(n)
        assert callable(fn) and inspect.signature(fn) == sig
    with pytest.raises(ValueError):
        deepnets.get('no_such_nets')
    with pytest.raises(ValueError):
        deepnets.get(None)
    assert deepnets.get('afm_nets')(None, None, None, None, None, None) is None      # fewer than 2 embeddings (deepnets.py:103)

    def custom(embeddings, flatten_emb_layer, dense_layer, concat_emb_dense, config, model_desc):
        return None
    assert deepnets.get_nets(['dnn_nets', custom, 'dnn_nets']) == ['dnn_nets', 'custom']
    assert deepnets.get('custom') is custom


def test_metainfo_records():
    from deeptables_b200.metainfo import CategoricalColumn, ContinuousColumn
    c = CategoricalColumn('x', 10000, 0)
    assert c.embeddings_output_dim == 10 and c.input_name == 'cat_x' and c.dtype == 'int32'
    assert hash(c) == hash('x')
    cc = ContinuousColumn('input_continuous_all', ['a', 'b', 'c'])
    assert cc.input_dim == 3 and cc.dtype == 'float32'


def test_preprocessor_conventions():
    from deeptables_b200 import deeptable
    from deeptables_b200.deeptable import DefaultPreprocessor
    df = pd.DataFrame({'a': ['x', 'y', None, 'x'], 'b': [1.0, np.nan, 3.0, 4.0], 'k': [7, 7, 7, 7]})
    pre = DefaultPreprocessor(deeptable.ModelConfig())
    X, y = pre.fit_transform(df, ['n', 'p', 'n', 'p'])
    assert pre.task == 'binary' and pre.labels == ['n', 'p'] and list(y) == [0, 1, 0, 1]
    assert [c.name for c in pre.categorical_columns] == ['a']
    assert pre.categorical_columns[0].vocabulary_size == 3 + 2        # nunique(+nan) + 2 (preprocessor.py:333)
    assert pre.continuous_columns[0].name == 'input_continuous_all' and pre.continuous_columns[0].column_names == ['b']
    assert 'k' not in X.columns                                        # auto_discard_unique
    assert not X['b'].isna().any()
    Xt = pre.transform_X(pd.DataFrame({'a': ['zzz'], 'b': [2.0], 'k': [7]}))
    assert int(Xt['a'][0]) == 3                                        # unseen -> reserved slot
    pre2 = DefaultPreprocessor(deeptable.ModelConfig())
    _, y2 = pre2.fit_transform(df, [0.5, 1.25, 3.75, 2.0])
    assert pre2.task == 'regression'


def test_ignore_case_dict():
    from deeptables_b200.deepmodel import IgnoreCaseDict
    d = IgnoreCaseDict({'AUC': 1, 'loss': 2})
    assert d['auc'] == 1 and 'Loss' in d
    d['Val_AUC'] = 3
    assert d['val_auc'] == 3
    with pytest.raises(KeyError):
        d[1]


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver times beside the GPU arm) runs without a GPU and
    prints one JSON line with the contract's keys."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--impl', 'reference', '--steps', '2',
                          '--warmup', '0', '--cpu-sample-rows', '128'], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line['impl'] == 'reference' and line['unit'] == 'rows/s' and line['value'] > 0
    for key in ('metric', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'config', 'cpu_baseline', 'e2e'):
        assert key in line, key
    assert line['e2e']['h2d_bytes_per_step'] == 0 and line['cpu_baseline']['kind'] in ('port', 'reference')
    assert line['steps'] == line['cpu_baseline']['steps'] == 2          # --steps is the number of steps timed
    assert line['warmup'] == 1                                           # the one untimed step it always runs
    out = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--impl', 'reference', '--dump-outputs', 'x'],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode != 0 and '--dump-outputs' in out.stderr


def test_ctypes_signatures_match_the_header_prototypes():
    """Every prototype in include/deeptables_b200.h against the ctypes table in _native.py: same arity and the
    same scalar class per argument (an ABI drift here corrupts arguments silently on the GPU box)."""
    import ctypes
    import re
    from deeptables_b200 import _native as nat
    with open(nat.HEADER_PATH) as f:
        text = re.sub(r'/\*.*?\*/', '', f.read(), flags=re.S)
    text = re.sub(r'//[^\n]*', '', text)
    protos = re.findall(r'([A-Za-z_][A-Za-z0-9_ \*]*?)\b(dtb_[a-z0-9_]+)\s*\(([^)]*)\)\s*;', text)
    assert len(protos) >= 30

    def classify_c(decl):
        decl = decl.strip()
        if '*' in decl:
            return 'ptr'
        base = re.sub(r'\b[A-Za-z_][A-Za-z0-9_]*$', '', decl).strip() or decl     # drop the parameter name
        base = base.replace('const', '').strip()
        return {'int': 'i32', 'int32_t': 'i32', 'int64_t': 'i64', 'long long': 'i64', 'size_t': 'u64',
                'unsigned long long': 'u64', 'uint64_t': 'u64', 'float': 'f32', 'double': 'f64'}[base]

    def classify_ct(t):
        if t in (ctypes.c_void_p, ctypes.c_char_p) or hasattr(t, 'contents') or getattr(t, '_type_', None) is ctypes.c_int and t is not ctypes.c_int:
            return 'ptr'
        return {ctypes.c_int: 'i32', ctypes.c_int64: 'i64', ctypes.c_longlong: 'i64', ctypes.c_size_t: 'u64',
                ctypes.c_ulonglong: 'u64', ctypes.c_float: 'f32', ctypes.c_double: 'f64'}[t]

    seen = set()
    for ret, name, args in protos:
        seen.add(name)
        assert name in nat._SIGNATURES, f'{name} declared in the header but not bound'
        res, argtypes = nat._SIGNATURES[name]
        params = [a for a in (x.strip() for x in args.split(',')) if a and a != 'void']
        assert len(params) == len(argtypes), f'{name}: header has {len(params)} parameters, ctypes table {len(argtypes)}'
        for k, (c_decl, ct) in enumerate(zip(params, argtypes)):
            assert classify_c(c_decl) == classify_ct(ct), f'{name} arg {k} ({c_decl!r}) bound as {ct}'
        ret = ret.replace('extern', '').replace('"C"', '').strip()
        want = 'ptr' if '*' in ret else ('void' if ret == 'void' else classify_c(ret + ' x'))
        got = 'void' if res is None else ('ptr' if res in (ctypes.c_char_p, ctypes.c_void_p) else classify_ct(res))
        assert want == got, f'{name}: return type {ret!r} bound as {res}'
    assert seen == set(nat._SIGNATURES), sorted(set(nat._SIGNATURES) ^ seen)


def test_cin_tc_set_variant_rejects_unknown_bits():
    """dtb_cin_tc_set_variant knows bits 0, 16 and 17 only: any other bit is an error that names the bit and
    leaves the flags as they were.  It touches no device."""
    from deeptables_b200 import _native as nat
    assert nat.lib.dtb_cin_tc_set_variant(1 | (1 << 12)) == -1          # DTB_ERR_INVALID_ARG
    assert 'bit 12' in nat.last_error()
    assert nat.lib.dtb_cin_tc_set_variant(1) == 0


def test_no_undefined_globals_in_gpu_only_code():
    """Function bodies of the host modules, bench.py and the GPU tests only execute on a GPU box; catch typos in
    global names here (the image has no pyflakes): tools/lint_names.py."""
    import glob
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location('lint_names', os.path.join(root, 'tools', 'lint_names.py'))
    lint = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(lint)
    files = (glob.glob(os.path.join(root, 'deeptables_b200', '*.py')) + glob.glob(os.path.join(root, 'tests', '*.py')) +
             glob.glob(os.path.join(root, 'tools', '*.py')) + [os.path.join(root, 'bench.py'), os.path.join(root, '__graft_entry__.py')])
    problems = [p for f in files for p in lint.check(f)]
    assert not problems, '\n'.join(problems)


def test_scope_param_stack_indices_and_f3_host_objects():
    """Host logic of the round-2 widening that needs no GPU: stacked parameter families (BilinearInteraction's per-pair
    matrices), per-model layer indices (fibi_nets / fg_nets), the focal-loss objects and the activation codes."""
    import torch
    from deeptables_b200 import layers, engine
    from deeptables_b200.deepmodel import _Scope
    scope = _Scope(torch.device('cpu'), 3)
    names = ['l/bilinear_weight0_1', 'l/bilinear_weight0_2', 'l/bilinear_weight1_2']
    w = scope.param_stack(names, (4, 4), 'glorot_uniform')
    assert tuple(w.shape) == (3, 4, 4) and scope.param_stack(names, (4, 4), 'glorot_uniform') is w
    assert scope.stacked == {'l/bilinear_weight0_1[*]': names}
    assert not torch.equal(w[0], w[1])                       # every slice is drawn on its own, with the fans of a (4, 4) matrix
    lim = (6.0 / 8) ** 0.5
    assert float(w.detach().abs().max()) <= lim
    with pytest.raises(ValueError):
        scope.param_stack(names, (4, 5), 'glorot_uniform')
    scope.param('l/bias', (3,), 'zeros')
    scope.freeze()
    assert scope.flat_p.numel() == 3 * 16 + 3 and scope.params['l/bilinear_weight0_1[*]'].grad is not None
    with pytest.raises(RuntimeError):
        scope.param_stack(['m/w0', 'm/w1'], (2, 2), 'zeros')
    assert (scope.next_index('senet_layer'), scope.next_index('senet_layer'), scope.next_index('concat_fgcnn_embedding')) == (0, 1, 0)
    scope._begin_pass()
    assert scope.next_index('senet_layer') == 0              # indices restart with every forward pass of the model
    fl = layers.BinaryFocalLoss(gamma=1.5, alpha=0.6)
    assert (fl.gamma, fl.alpha) == (1.5, 0.6) and fl.get_config()['gamma'] == 1.5
    assert isinstance(layers.CategoricalFocalLoss(), layers.BinaryFocalLoss)
    with pytest.raises(NotImplementedError):
        layers.GHMCLoss()
    with pytest.raises(NotImplementedError):
        layers.VarLenColumnEmbedding(3, 4, 'uniform', None, None)
    assert engine.ACT_CODES == {None: 0, 'linear': 0, 'relu': 1, 'tanh': 2}
    assert engine.BILINEAR_TYPES == {'field_all': 0, 'field_each': 1, 'field_interaction': 2}
    g = torch.Generator().manual_seed(0)
    t = layers.init_tensor((64, 32), 'glorot_normal', 'cpu', g)
    std = (2.0 / 96) ** 0.5 / 0.87962566103423978
    assert float(t.abs().max()) <= 2 * std + 1e-6 and abs(float(t.std()) - (2.0 / 96) ** 0.5) < 0.01
