#!/usr/bin/env python
"""bench.py -- xDeepFM train-step throughput on synthetic Criteo-shape rows (BASELINE.json metric).

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the CPU baseline arm (oracle port; TF is not installable)
    python bench.py ... --dump-outputs DIR    # also write the last timed step's outputs as DIR/<name>.npy

A "step" = one full optimiser step (forward + loss + backward + DP exchange + Adam) of xDeepFM
(`linear + cin_nets + dnn_nets`, CIN 128x128x128) on one batch of 65 536 rows per GPU: 13 dense +
26 sparse fields, vocab 1 M per field, embed_dim 16 (BASELINE.json configs[2]).  Weak scaling: the
per-GPU batch is fixed.  One JSON line is printed by rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

F_FIELDS, N_DENSE = 26, 13
CIN_SIZES = (128, 128, 128)
_CIN = {'cross_layer_size': CIN_SIZES, 'activation': 'relu', 'use_residual': False, 'use_bias': False, 'direct': False,
        'reduce_D': False}
# BASELINE.json configs[1..4] (configs[0], the bank-data README example, needs hypernets' data set: tests/ cover it)
CONFIGS = {
    'xdeepfm': dict(nets=['linear', 'cin_nets', 'dnn_nets'], dim=16, batch=65536, kw={'cin_params': _CIN},
                    metric='xDeepFM train rows/sec, Criteo-shape synthetic',
                    workload='xDeepFM (linear+cin_nets+dnn_nets) train step, CIN 128x128x128 direct=False, 13 dense + 26 '
                             'sparse fields, vocab 1M/field, embed_dim 16 (BASELINE configs[2])'),
    'deepfm_bs8192': dict(nets=['linear', 'fm_nets', 'dnn_nets'], dim=16, batch=8192, kw={},
                          metric='DeepFM train rows/sec, Criteo-shape synthetic',
                          workload='DeepFM (linear+fm_nets+dnn_nets) train step, 13 dense + 26 sparse fields, vocab '
                                   '1M/field, embed_dim 16, bs 8192 (BASELINE configs[1])'),
    'dcn6_autoint4x32': dict(nets=['dcn_nets', 'autoint_nets'], dim=32, batch=65536,
                             kw={'cross_params': {'num_cross_layer': 6},
                                 'autoint_params': {'num_attention': 3, 'num_heads': 4, 'dropout_rate': 0,
                                                    'use_residual': True}},
                             metric='DCN(6)+AutoInt(4 heads, d=32) train rows/sec, Criteo-shape synthetic',
                             workload='dcn_nets (CrossNet depth 6 + DNN) stacked with autoint_nets (3 layers, 4 heads, '
                                      'd=32) train step, 13 dense + 26 sparse fields, vocab 1M/field, embed_dim 32 '
                                      '(BASELINE configs[3])'),
    'five_nets': dict(nets=['fm_nets', 'cin_nets', 'cross_nets', 'autoint_nets', 'pnn_nets'], dim=16, batch=16384,
                      kw={'cin_params': _CIN},
                      metric='five-net mix train rows/sec, Criteo-shape synthetic',
                      workload="nets=['fm_nets','cin_nets','cross_nets','autoint_nets','pnn_nets'] train step, 13 dense + 26 "
                               'sparse fields, vocab 1M/field, embed_dim 16, 131072 global rows / 8 GPUs = 16384 per GPU '
                               '(BASELINE configs[4])'),
}
EMB_DIM = 16      # of the headline config (CIN_FLOP_PER_ROW below)
# algorithmic work per row, SURVEY.md 8(d) / DESIGN.md section 5
CIN_FLOP_PER_ROW = 2 * EMB_DIM * sum(l * k for l, k in zip(CIN_SIZES, (26 * 26, 26 * 64, 26 * 64)))  # 16 400 384
CIN_BYTES_PER_ROW = 4 * F_FIELDS + 4 * F_FIELDS * EMB_DIM + 4 * (64 + 64 + 128)                        # ids + rows + pooled


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20, help='timed steps of every timed loop (at least 1)')
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--config', default='xdeepfm', choices=sorted(CONFIGS),
                    help='which BASELINE.json config to run (default: configs[2], the headline)')
    ap.add_argument('--batch', type=int, default=0, help='rows per GPU per step (default: the config\'s)')
    ap.add_argument('--vocab', type=int, default=1_000_000)
    ap.add_argument('--cpu-sample-rows', type=int, default=4096)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--cin-precision', type=int, default=0)
    ap.add_argument('--no-graph', action='store_true', help='eager launches instead of the CUDA-graph replay of the train step')
    ap.add_argument('--cin-exp', type=int, default=0,
                    help='profiling only: experiment build of the CIN backward kernels (cin_tc.cu), 0 = product kernels')
    ap.add_argument('--id-dist', default='uniform', choices=['uniform', 'zipf'],
                    help="categorical id distribution of the synthetic batches (the headline is 'uniform')")
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed train step computed to DIR/<name>.npy (rank 0), so that two builds '
                         'can be compared output for output on the same seeded inputs (b200 arm only)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the b200 arm; --impl reference has none to write')
    return args


def config_overrides(name, cin_precision=0):
    """ModelConfig fields of a bench config as a plain dict (no package import: the reference arm uses it too)."""
    spec = CONFIGS[name]
    d = dict(nets=list(spec['nets']), embeddings_output_dim=spec['dim'], embedding_dropout=0, dense_dropout=0,
             metrics=['AUC'])
    for k, v in spec['kw'].items():
        d[k] = dict(v)
    if 'cin_params' in d and cin_precision:
        d['cin_params']['precision'] = cin_precision
    return d


def make_config(name='xdeepfm', cin_precision=0):
    from deeptables_b200 import deeptable
    return deeptable.ModelConfig(**config_overrides(name, cin_precision))


def reference_config(name):
    """The same configuration for the CPU arm WITHOUT importing the product package (whose import loads the CUDA
    library): the reference's own ModelConfig() defaults, as dumped from /root/reference by
    tests/golden/make_reference_golden.py, overlaid with the bench overrides.  oracle/model_ref.py reads dicts."""
    with open(os.path.join(ROOT, 'tests', 'golden', 'reference_modelconfig.json')) as f:
        conf = dict(json.load(f)['defaults'])
    conf.update(config_overrides(name))
    return conf


def synth_batches(n_batches, batch, vocab, seed, id_dist='uniform', pin=True):
    """Synthetic Criteo-shape rows (BASELINE.md section 3): ids uniform in [0, vocab) (or, labelled, the
    Zipf(1.05) variant of SURVEY 8d: rank r drawn with p ~ r^-1.05, many duplicate rows per batch), dense N(0,1),
    label Bernoulli(0.25).  Returned as pinned HOST tensors."""
    import torch
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n_batches):
        if id_dist == 'zipf':
            # inverse-CDF sampling of a truncated Zipf(1.05) over ranks 1..vocab (continuous approximation)
            a = 1.05
            u = torch.rand(batch, F_FIELDS, generator=g, dtype=torch.float64)
            top = float(vocab + 1) ** (1.0 - a)
            r = (1.0 + u * (top - 1.0)) ** (1.0 / (1.0 - a))
            idx = (r.floor().clamp_(1, vocab) - 1).to(torch.int32)
        else:
            idx = torch.randint(0, vocab, (batch, F_FIELDS), generator=g, dtype=torch.int32)
        dense = torch.randn(batch, N_DENSE, generator=g)
        y = (torch.rand(batch, 1, generator=g) < 0.25).float()
        out.append(tuple(t.pin_memory() if (pin and torch.cuda.is_available()) else t for t in (idx, dense, y)))
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.samples, self._stop, self._t = index, [], threading.Event(), None

    def _run(self):
        # fast path: NVML in-process (a sample every 20 ms, so even a 0.2 s timed region gets ~10 of them); any failure
        # falls back to spawning nvidia-smi (one sample per ~0.3 s).  Both produce the same 7-field sample.
        nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            nv = (pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.index))
        except Exception:
            nv = None
        while nv is not None and not self._stop.is_set():
            try:
                ml, h = nv
                sm = ml.nvmlDeviceGetClockInfo(h, ml.NVML_CLOCK_SM)
                mx = ml.nvmlDeviceGetMaxClockInfo(h, ml.NVML_CLOCK_SM)
                getter = getattr(ml, 'nvmlDeviceGetCurrentClocksEventReasons', None) or \
                    ml.nvmlDeviceGetCurrentClocksThrottleReasons
                r = int(getter(h))
                flag = lambda bit: 'Active' if r & bit else 'Not Active'        # noqa: E731
                # NVML reason bits: SwPowerCap 0x4, HwSlowdown 0x8, SwThermalSlowdown 0x20, HwThermalSlowdown 0x40
                self.samples.append([str(sm), str(mx), '', flag(0x8), flag(0x40), flag(0x20), flag(0x4)])
            except Exception:
                nv = None
                break
            self._stop.wait(0.02)
        while not self._stop.is_set():
            try:
                out = subprocess.run(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                      '-i', str(self.index)], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(',')]
                if len(parts) >= 7:
                    self.samples.append(parts)
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace('.', '').isdigit())
        mx = [float(s[1]) for s in self.samples if s[1].replace('.', '').isdigit()]
        reasons = set()
        for s in self.samples:
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), s[3:7]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(self.samples)}


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {'hbm_gbs': p['hbm_gbs'], 'bf16_tflops': p['bf16_tflops'],
                'bf16_tflops_sustained': p.get('bf16_tflops_sustained', p['bf16_tflops']), 'source': 'measured'}
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0, 'source': 'fallback'}


def cpu_baseline(args, conf, steps, warmup=1):
    """The reference's CPU path: TF/Keras cannot be installed here, so this is the oracle PORT (torch CPU fp32
    restatement of the identical graph) on the host cores, on a bounded sample of the same workload: one micro-batch
    of `--cpu-sample-rows` rows of the config's batch (the reference formulation materialises 7 GB per CIN layer at
    65 536 rows), table rows capped at 100 k per field (per-row work does not depend on the table size).
    Exactly `steps` train steps are timed, after `warmup` (at least one) untimed ones."""
    import torch
    from oracle import model_ref as M
    spec = CONFIGS[args.config]
    dim = spec['dim']
    cores = os.cpu_count() or 1
    rows = min(args.cpu_sample_rows, spec['batch'])
    vocab = min(args.vocab, 100_000)
    state = M.init_state(conf, [vocab] * F_FIELDS, [dim] * F_FIELDS, N_DENSE, seed=1234)
    tr = M.RefTrainer(state, conf, F_FIELDS)
    (idx, dense, y), = synth_batches(1, rows, vocab, 99, pin=False)
    # the graph is dominated by memory-bound elementwise ops: on many-core hosts "all cores" is often not the fastest
    # setting, so both are reported: a calibration over thread counts on a small slice picks the one that is timed,
    # and the all-cores time of the same slice is given next to it
    cal_rows = min(rows, 512)
    cal = {}
    for nt in sorted({c for c in (8, 16, 32, 64, cores) if c <= cores}):
        torch.set_num_threads(nt)
        tr.train_step(idx[:cal_rows], dense[:cal_rows], y[:cal_rows, 0])
        t0 = time.perf_counter()
        tr.train_step(idx[:cal_rows], dense[:cal_rows], y[:cal_rows, 0])
        cal[nt] = time.perf_counter() - t0
    threads = min(cal, key=cal.get)
    torch.set_num_threads(threads)
    warmup = max(1, warmup)
    for _ in range(warmup):
        tr.train_step(idx, dense, y[:, 0])
    t0 = time.perf_counter()
    for _ in range(steps):
        tr.train_step(idx, dense, y[:, 0])
    dt = (time.perf_counter() - t0) / steps
    return {'value': rows / dt, 'unit': 'rows/s', 'cores': threads, 'kind': 'port', 'steps': steps, 'warmup': warmup,
            'sample': f'{steps} train steps x {rows} rows (one micro-batch of the {spec["batch"]}-row batch), {threads} threads = '
                      f'fastest of a calibration over {sorted(cal)} on {cores} host cores (all {cores} cores: '
                      f'{cal[max(cal)] / cal[threads]:.2f}x slower on the calibration slice), {args.config}, vocab '
                      f'{vocab}/field, torch-CPU fp32 oracle port (TensorFlow not installable: no network)',
            'sec_per_step': dt}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    spec = CONFIGS[args.config]
    conf = reference_config(args.config)              # plain dict: nothing of the product package is imported
    base = cpu_baseline(args, conf, args.steps, args.warmup)
    assert 'deeptables_b200' not in sys.modules, 'the reference arm must not load the product library'
    line = {'impl': 'reference', 'metric': spec['metric'], 'value': base['value'],
            'unit': 'rows/s', 'n_gpus': args.gpus, 'steps': base['steps'], 'warmup': base['warmup'],
            'ms_per_step': base['sec_per_step'] * 1e3, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': spec['workload'] + '; CPU sample', 'global_batch': min(args.cpu_sample_rows, spec['batch'])},
            'cpu_baseline': {k: base[k] for k in ('value', 'unit', 'cores', 'kind', 'steps', 'sample')},
            'e2e': {'value': base['value'], 'unit': 'rows/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line))


def _timed_alone(fn, flush):
    """Median of 5 launches timed with CUDA events on the launching stream, L2 evicted by reading a 512 MB buffer."""
    import torch
    for _ in range(2):
        fn()
    times = []
    for _ in range(5):
        flush.sum()                                # read > L2 of clean lines: nothing cache-resident, nothing dirty to write back
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1) * 1e-3)
    return sorted(times)[len(times) // 2]


def time_fm_linear_kernel(model, cat, dense, peaks):
    """configs[1] (DeepFM): the fused gather + linear + FM forward, HBM-bound: 104 B ids + 1 664 B rows + 52 B dense +
    8 B out per row (SURVEY 8d)."""
    import torch
    from deeptables_b200 import _native as N
    from deeptables_b200._native import ptr
    t = model.table
    b = cat.shape[0]
    w_lin = model._scope.params['linear/kernel'].detach().reshape(-1).contiguous() if 'linear/kernel' in model._scope.params \
        else torch.zeros(F_FIELDS + N_DENSE, device=cat.device)
    o1, o2 = torch.empty(b, 1, device=cat.device), torch.empty(b, 1, device=cat.device)
    flush = torch.zeros(512 << 20, dtype=torch.uint8, device=cat.device)

    def fwd():
        N.check(N.lib.dtb_fm_linear_fwd(ptr(cat), ptr(t.weight), ptr(t.row_offsets), ptr(dense), ptr(w_lin), ptr(o1), ptr(o2), b,
                                        F_FIELDS, t.dim, N_DENSE, None, N.stream_ptr()), 'fm_linear_fwd')
    dt = _timed_alone(fwd, flush)
    bytes_row = 4 * F_FIELDS + 4 * F_FIELDS * t.dim + 4 * N_DENSE + 8
    gbs = b * bytes_row / dt / 1e9
    return {'bound': 'hbm', 'achieved': gbs, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': gbs / peaks['hbm_gbs'],
            'traffic': None, 'kernel': 'fm_linear_fwd (gather + linear + FM fused)', 'ms': dt * 1e3,
            'algorithmic_bytes_per_launch': b * bytes_row, 'peak_source': peaks['source']}


def time_attention_kernel(model, cat, peaks, heads):
    """configs[3]: one MultiheadAttention core launch (softmax(QK^T/sqrt(dh))V + residual, relu) on [B, F, 4D]
    projections, HBM-bound at ~5 FLOP/B: reads 4*F*D, writes F*D floats per row."""
    import torch
    from deeptables_b200 import _native as N
    from deeptables_b200._native import ptr
    b, d = cat.shape[0], model.table.dim
    qkvr = torch.randn(b, F_FIELDS, 4 * d, device=cat.device)
    y = torch.empty(b, F_FIELDS, d, device=cat.device)
    flush = torch.zeros(512 << 20, dtype=torch.uint8, device=cat.device)

    def fwd():
        N.check(N.lib.dtb_attention_core_fwd(ptr(qkvr), ptr(y), b, F_FIELDS, d, heads, 1, N.stream_ptr()), 'attention_core_fwd')
    dt = _timed_alone(fwd, flush)
    bytes_row = 4 * F_FIELDS * d * 5
    gbs = b * bytes_row / dt / 1e9
    return {'bound': 'hbm', 'achieved': gbs, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': gbs / peaks['hbm_gbs'],
            'traffic': None, 'kernel': f'attention_core_fwd ({heads} heads, d={d})', 'ms': dt * 1e3,
            'algorithmic_bytes_per_launch': b * bytes_row, 'peak_source': peaks['source']}


def time_cin_kernel(model, cat, peaks):
    """Roofline of the dominant kernel family: the CIN forward kernel exactly as the train step runs it
    (training mode: activations saved), timed alone with CUDA events on its stream, L2 flushed between
    launches; plus the CIN backward (dgrad + 3 wgrad launches) for information."""
    import torch
    from deeptables_b200 import _native as N
    from deeptables_b200._native import ptr
    t = model.table
    b = cat.shape[0]
    sizes_c = N.int_array(CIN_SIZES)
    weights = torch.cat([model._scope.params[f'cin/f_{k}'].detach().reshape(-1) for k in range(3)]).contiguous()
    pooled = torch.empty(b, 256, device=cat.device)
    d_pooled = torch.randn(b, 256, device=cat.device) * 1e-3
    ws_bytes = N.lib.dtb_cin_workspace_bytes(b, F_FIELDS, EMB_DIM, sizes_c, 3, 0, 1)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=cat.device)
    saved = torch.empty(N.lib.dtb_cin_saved_bytes(b, F_FIELDS, EMB_DIM, sizes_c, 3, 0), dtype=torch.uint8, device=cat.device)
    dw = torch.zeros_like(weights)
    flush = torch.zeros(512 << 20, dtype=torch.uint8, device=cat.device)
    precision = model.config.cin_params.get('precision', 0)
    t.ensure_training_state()

    def fwd():
        N.check(N.lib.dtb_cin_fwd(ptr(cat), ptr(t.weight), ptr(t.row_offsets), ptr(weights), None, ptr(pooled), ptr(saved),
                                  ptr(ws), ws_bytes, b, F_FIELDS, EMB_DIM, sizes_c, 3, 0, 1, precision, None,
                                  N.stream_ptr()), 'cin_fwd')

    def bwd():
        N.check(N.lib.dtb_cin_bwd(ptr(cat), ptr(t.weight), ptr(t.row_offsets), ptr(weights), ptr(d_pooled), ptr(saved),
                                  ptr(t.grad), ptr(dw), None, ptr(ws), ws_bytes, b, F_FIELDS, EMB_DIM, sizes_c, 3, 0, 1,
                                  precision, N.stream_ptr()), 'cin_bwd')

    dt = _timed_alone(fwd, flush)
    dt_b = _timed_alone(bwd, flush)
    t.grad.zero_()                                     # the probe's gradients must not leak into training
    mode = N.lib.dtb_cin_resolved_precision(F_FIELDS, EMB_DIM, sizes_c, 3, 0, precision)     # what 'auto' runs for this shape
    tc = mode in (2, 3, 4)
    tf = b * CIN_FLOP_PER_ROW / dt / 1e12
    kname = {4: 'cin_tc2_fwd_kernel', 2: 'cin_tc_fwd_kernel', 3: 'cin_tc_fwd_kernel'}.get(mode)
    traffic = None
    tpath = os.path.join(ROOT, 'profiles', 'r2_cin_tc_traffic.json')
    if kname and os.path.exists(tpath) and b == 65536:
        with open(tpath) as f:
            tj = json.load(f).get(kname)            # ncu --set full capture of this kernel at this shape (training mode)
        if tj:
            traffic = tj['dram_bytes_read'] + tj['dram_bytes_write']
    return {'bound': 'tensor', 'achieved': tf, 'peak': peaks['bf16_tflops'], 'unit': 'TFLOP/s',
            'frac': tf / peaks['bf16_tflops'], 'traffic': traffic,
            'kernel': {4: 'cin_tc2_fwd_kernel (tcgen05, ONE pass on power-of-two-scaled fp16 operands, two threads per GEMM row)',
                       2: 'cin_tc_fwd_kernel (tcgen05, bf16x3 split: 3 tensor passes per algorithmic FLOP)',
                       3: 'cin_tc_fwd_kernel (tcgen05, one bf16 pass)'}.get(mode, 'cin_fwd (any-shape formulation, dense_tc GEMMs)'),
            'ms': dt * 1e3, 'algorithmic_flop_per_launch': b * CIN_FLOP_PER_ROW,
            'algorithmic_bytes_per_launch': b * CIN_BYTES_PER_ROW,
            'executed_tensor_tflops': tf * (3 if mode == 2 else 1),
            'hbm_gbs_informational': b * CIN_BYTES_PER_ROW / dt / 1e9, 'peak_source': peaks['source'],
            'cin_backward': {'ms': dt_b * 1e3, 'algorithmic_tflops': 2 * b * CIN_FLOP_PER_ROW / dt_b / 1e12,
                             'kernels': 'cin_tc2_dgrad_kernel + 3 x cin_tc2_wgrad_kernel' if mode == 4 else
                                        'cin_tc_dgrad_kernel + 3 x cin_tc_wgrad_kernel'}}


DUMP_EMB_SAMPLES = 65536          # (row, field) ids of the last batch whose embedding rows --dump-outputs writes
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(model, prob, cat, out_dir):
    """Write what one train step hands its caller, right after that step: the batch predictions it returns, the summed
    loss it accumulates (over every step since the model was built), the dense parameters and buffers after the Adam
    update, and the embedding rows of a fixed, seeded sample of the batch's ids.  Only rows the step touched are
    sampled: with lazy Adam the rest of the table is brought up to date only when it is next read.  When the predictions
    of a large --batch would take the files past DUMP_MAX_BYTES, a fixed, seeded sample of their rows is written, in
    row order.  Float atomics in the gradient reductions make two runs agree to round-off grown by the training steps,
    not bit for bit: two runs with the default arguments (5 warm-up + 20 timed xDeepFM steps), compared file by file,
    gave predictions within 1.2e-3 of each other on one B200 at its 1000 W power limit."""
    import numpy as np
    import torch
    t, scope = model.table, model._scope
    g = torch.Generator().manual_seed(0)
    pos = torch.randint(0, cat.numel(), (min(DUMP_EMB_SAMPLES, cat.numel()),), generator=g).to(cat.device)
    rows = cat.reshape(-1)[pos].long() + t.row_offsets[pos % cat.shape[1]]
    arrays = {'loss_sum': model._loss_acc.double(), 'dense_params': scope.flat_p,
              'embedding_rows': t.weight.index_select(0, rows)}
    if scope.buffers:
        arrays['dense_buffers'] = torch.cat([b.reshape(-1).float() for b in scope.buffers.values()])
    room = (DUMP_MAX_BYTES - sum(v.numel() * v.element_size() for v in arrays.values())) // (4 * prob[0].numel())
    if prob.shape[0] > room:
        keep = torch.randperm(prob.shape[0], generator=g)[:room].sort().values.to(prob.device)
        prob = prob.index_select(0, keep)
    arrays['predictions'] = prob.float()
    arrays = {k: v.detach().cpu().numpy() for k, v in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f'{k}.npy'), a)


def main():
    args = parse_args()
    if args.impl == 'reference':
        run_reference(args)
        return
    if args.no_graph:
        os.environ['DTB_CUDA_GRAPH'] = '0'
    import torch
    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    from deeptables_b200 import _native as N
    from deeptables_b200.deepmodel import DeepModel
    from deeptables_b200.metainfo import CategoricalColumn, ContinuousColumn

    spec = CONFIGS[args.config]
    if not args.batch:
        args.batch = spec['batch']
    emb_dim = spec['dim']
    conf = make_config(args.config, args.cin_precision)
    if args.cin_exp:
        N.check(N.lib.dtb_cin_tc_set_variant(1 | (args.cin_exp << 12)), 'cin_tc_set_variant')
    cats = [CategoricalColumn(f'C{i + 1}', args.vocab, emb_dim) for i in range(F_FIELDS)]
    conts = [ContinuousColumn('input_continuous_all', [f'I{i + 1}' for i in range(N_DENSE)])]
    model = DeepModel('binary', 2, conf, cats, conts, seed=1234)
    model._build_model()
    # a fresh batch every step (warm-up and timed steps alike): with a small rotating pool every embedding row would be
    # re-touched after a few steps and the exact-lazy Adam catch-up would never replay more than that many steps
    n_pool = min(max(args.warmup, 3) + args.steps, 64)
    host = synth_batches(n_pool, args.batch, args.vocab, 1234 + rank, args.id_dist)
    devb = [tuple(t.cuda(non_blocking=True) for t in hb) for hb in host]
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for s in range(steps):
            fn(s)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device='cuda')
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) * 1e-3

    last = {}

    def dev_step(s):
        c, d, y = devb[s % n_pool]
        last['prob'] = model.train_step(c, d, y)

    def e2e_step(s):
        c, d, y = host[s % n_pool]
        model.train_on_batch(c, d, y)            # H2D of the batch + D2H of the loss inside

    for s in range(max(args.warmup, 3)):
        dev_step(s)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = N.lib.dtb_launch_count()
    secs = timed(dev_step, args.steps)
    launches = N.lib.dtb_launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # before the e2e steps below train the model further (and, under a CUDA graph, overwrite the same predictions)
        dump_outputs(model, last['prob'], devb[(args.steps - 1) % n_pool][0], args.dump_outputs)
    for s in range(2):
        e2e_step(s)
    secs_e2e = timed(e2e_step, args.steps)
    loss = float(model._loss_acc.item()) / args.batch

    # score-only pass (SURVEY 8d "also report score-only"): forward + task activation, device-resident inputs,
    # no collective.  Informational: a failure here must never cost the headline line.
    score = None
    try:
        def score_step(s):
            c, d, _ = devb[s % n_pool]
            model.predict_step(c, d)
        for s in range(2):
            score_step(s)
        secs_score = timed(score_step, args.steps)
        score = {'value': args.batch * world * args.steps / secs_score, 'unit': 'rows/s',
                 'ms_per_step': secs_score / args.steps * 1e3, 'what': 'DeepModel.predict_step, inputs resident in HBM'}
    except Exception as exc:                                # pragma: no cover
        score = {'error': f'{type(exc).__name__}: {exc}'[:200]}

    if rank == 0:
        peaks = measured_peaks()
        if 'cin_nets' in spec['nets']:
            roof = time_cin_kernel(model, devb[0][0], peaks)
        elif 'autoint_nets' in spec['nets']:
            roof = time_attention_kernel(model, devb[0][0], peaks, spec['kw']['autoint_params']['num_heads'])
        else:
            roof = time_fm_linear_kernel(model, devb[0][0], devb[0][1], peaks)
        rows = args.batch * world * args.steps
        h2d = sum(t.numel() * t.element_size() for t in host[0])
        line = {
            'metric': spec['metric'], 'value': rows / secs, 'unit': 'rows/s',
            'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': secs / args.steps * 1e3,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': ('f32 storage and accumulation; CIN GEMMs: one tcgen05 pass on power-of-two-scaled fp16 operands (error ~2e-4 '
                      'of the output scale); Dense GEMMs: bf16x3 split' if roof['kernel'].startswith('cin_tc2')
                      else 'f32 (CIN GEMMs: bf16x3 split on tcgen05, fp32 accumulate)' if roof['kernel'].startswith('cin_tc_')
                      else 'f32 (Dense GEMMs: bf16x3 split on tcgen05, fp32 accumulate)'),
            'experiment_build': args.cin_exp or None,
            'data': 'synthetic' if args.id_dist == 'uniform' else f'synthetic ({args.id_dist} ids: NOT the headline distribution)',
            'config': {'workload': spec['workload'], 'name': args.config,
                       'global_batch': args.batch * world, 'per_gpu_batch': args.batch, 'parallelism': f'dp{world}',
                       'optimizer': 'Adam(1e-3): dense weights dense, embedding rows exact-lazy (bit-identical to '
                                    'dense Keras Adam)', 'embedding_dropout': 0,
                       'batches': f'{n_pool} distinct synthetic batches, one per step (fresh ids every step)',
                       'l2_policy': 'inputs larger than L2: 1.66 GB tables + a distinct batch per step (7 MB ids each); '
                                    'roofline kernel timing evicts L2 by reading a 512 MB buffer between launches'},
            'e2e': {'value': rows / secs_e2e, 'unit': 'rows/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 8,
                    'ms_per_step': secs_e2e / args.steps * 1e3},
            'gpu_launches': int(launches),
            'cuda_graph': bool(getattr(model, '_graphs', None)) and not getattr(model, '_graph_failed', False),
            'roofline': roof, 'clocks': clocks, 'final_loss': loss,
            'score_only': score,
        }
        if world == 1 and not args.no_cpu_baseline:
            base = cpu_baseline(args, reference_config(args.config), args.steps)
            line['cpu_baseline'] = {k: base[k] for k in ('value', 'unit', 'cores', 'kind', 'steps', 'sample')}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
