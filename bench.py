#!/usr/bin/env python
"""Benchmark of the NLT UV-space hot path (BASELINE.json metric: UV texels/sec fwd+bwd @1024^2 x 64ch).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K ...  # reference arithmetic on the host CPU cores
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/<name>.npy

A "step" is one full training pass of the hot path over one synthetic batch: Model.call (fused input gather +
two-stream U-Net + UV->camera tail), L2 loss, full backward to every weight gradient, (N>1: the gradient all-reduce
over NCCL, overlapped with backward) and the fused AMSGrad update -- all of it one CUDA-graph replay per step.

Workloads (SURVEY.md 8d; `--workload`, default cfg4 = the configuration the metric is quoted on):
  cfg4    synthetic 64-channel query stack (base 3 + cvis 1 + lvis 1 + 59 extra maps), 1024^2 UV, depth 256, k2 s2,
          batch 8 PER GPU (weak scaling; N = 4 is BASELINE's global batch 32); `--scaling strong` = global batch 32
  cfg4k3  the same with 3x3 kernels (the north star's "3x3xC contraction")
  cfg2    dragon_specular as shipped (5-channel query stack), 1024^2, batch 8
  cfg3    dragon_sss (depth 1024), 6-neighbour observed-light stack, 1024^2, batch 16
  cfg1    dragon_specular 256^2, ONE view x light, forward only through the cached observation features (nlt_test)
The default N = 1 run prints the cfg4 line and carries the others (plus cfg4 at batch 1 and 32) as sub-records under
`extra`; N > 1 adds the strong-scaling record.  One JSON line on stdout (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, 'neural-light-transport_b200')
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = 'UV texels/sec fwd+bwd'
UNIT = 'texels/s'

# SURVEY.md 8(d): block-granularity algorithmic HBM bytes per texel (fwd, fwd+bwd) and conv FLOPs per texel (fwd)
WORKLOADS = {
    'cfg4': dict(uv=1024, c_extra=59, depth=256, kernel=2, k_obs=1, batch=8, train=True, bytes=(1102.0, 2918.0),
                 flop_fwd=15352.0,
                 desc='cfg4: synthetic 64-channel query stack (base 3 + cvis 1 + lvis 1 + 59 extra), dragon_specular '
                      'net (depth0 16, depth 256, k2 s2, leakyrelu, K=1 obs)'),
    'cfg4k3': dict(uv=1024, c_extra=59, depth=256, kernel=3, k_obs=1, batch=8, train=True, bytes=(1102.0, 2918.0),
                   flop_fwd=31592.0, desc='cfg4 with 3x3 kernels (k3 s2)'),
    'cfg2': dict(uv=1024, c_extra=0, depth=256, kernel=2, k_obs=1, batch=8, train=True, bytes=(866.0, 2210.0),
                 flop_fwd=13464.0, desc='cfg2: dragon_specular net (depth0 16, depth 256, k2 s2, leakyrelu, K=1 obs)'),
    'cfg3': dict(uv=1024, c_extra=0, depth=1024, kernel=2, k_obs=6, batch=16, train=True, bytes=(1888.0, 4798.0),
                 flop_fwd=47864.0, desc='cfg3: dragon_sss net (depth 1024, 18 layers), K=6 observed-light stack'),
    'cfg1': dict(uv=256, c_extra=0, depth=256, kernel=2, k_obs=1, batch=1, train=False, bytes=(866.0, 2210.0),
                 flop_fwd=13464.0,
                 desc='cfg1: dragon_specular net, single view x light, forward only with cached observation '
                      'features (nlt_test.py semantics)'),
}


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d['hbm_gbs']), float(d.get('bf16_tflops_sustained', d.get('bf16_tflops', 1400.0))), 'measured'
    return 6650.0, 1400.0, 'fallback'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self.thread = None

    def start(self):
        def run():
            q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
                 'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
            while not self._stop.is_set():
                try:
                    out = subprocess.check_output(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q,
                                                   '--format=csv,noheader,nounits'], timeout=5).decode()
                    self.rows.append([x.strip() for x in out.strip().split(',')])
                except Exception:
                    pass
                self._stop.wait(0.1)
        self.thread = threading.Thread(target=run, daemon=True)
        self.thread.start()

    def stop(self):
        self._stop.set()
        if self.thread:
            self.thread.join(timeout=10)
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({names[i] for r in self.rows for i in range(4) if len(r) > 2 + i and r[2 + i] == 'Active'})
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(sm)}


def make_config(wl):
    from util import io as ioutil
    return ioutil.make_config(uvh=wl['uv'], uvw=wl['uv'], imh=wl['uv'], imw=wl['uv'], loss='l2', depth0=16,
                              depth=wl['depth'], kernel=wl['kernel'], stride=2)


def oracle_cfg(wl):
    uv = wl['uv']
    return dict(depth0=16, depth=wl['depth'], kernel=wl['kernel'], stride=2, norm='None', act='leakyrelu', pool='None',
                use_obs=True, skip_connect_base=True, imh=uv, imw=uv, uvh=uv, uvw=uv)


def workload_config(wl_name, wl, batch, world, scaling, graph=True):
    uv = wl['uv']
    return {'workload': '%s, %dx%d UV, %dx%d camera, batch %d per GPU, %s' % (
                wl['desc'], uv, uv, uv, uv, batch, 'fwd+L2+bwd+AMSGrad' if wl['train'] else 'forward only'),
            'name': wl_name, 'query_channels': 5 + wl['c_extra'], 'observations': wl['k_obs'],
            'kernel': wl['kernel'], 'depth': wl['depth'], 'global_batch': batch * world, 'uv': uv,
            'parallelism': 'dp%d' % world, 'scaling': scaling, 'cuda_graph': graph,
            'l2_flush': 'inputs+activations per step (GBs) exceed the 126 MB L2; fresh batch buffers rotate'}


# ----------------------------------------------------------------------------
# reference arm: the restated reference arithmetic on the host CPU cores
# ----------------------------------------------------------------------------
def cpu_reference_step_fn(wl, batch):
    """Returns (fn, texels_per_call): one pass of the oracle (torch CPU, fp32) over `batch` samples: fwd+bwd for the
    training workloads, forward through the observation-feature override for cfg1."""
    from oracle import nlt_oracle as O
    from util import synth
    uv = wl['uv']
    cfg = oracle_cfg(wl)
    params = O.init_params(cfg, c_query=5 + wl['c_extra'], seed=7, dtype=torch.float32)
    bt = synth.make_batch(batch, uv, uv, seed=1235, c_extra=wl['c_extra'], k_obs=wl['k_obs'])
    if not wl['train']:
        with torch.no_grad():
            feat = O.extract_feat(params, cfg, [(bt[1], bt[5])])

        def fwd():
            with torch.no_grad():
                pred = O.model_call(params, cfg, bt, 'test', obs_override=[f.expand(batch, -1, -1, -1) for f in feat])[0]
            return float(pred.mean())
        return fwd, batch * uv * uv
    for v in params.values():
        v.requires_grad_(True)

    def fn():
        for v in params.values():
            v.grad = None
        loss = O.train_loss(params, cfg, bt, batch)
        loss.backward()
        return float(loss.detach())
    return fn, batch * uv * uv


def calibrate_cpu_threads(wl, batch):
    """Many-core hosts run this conv stack SLOWER with one torch thread per logical core (oversubscribed oneDNN
    primitives on 16-channel tensors), so the CPU arm picks the thread count that maximises ITS OWN throughput --
    probed at the measured size -- and reports it as `cores`.  Returns (cores, fn, texels, seconds of the best probe)."""
    cores = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, cores) if c <= cores})
    fn, texels = cpu_reference_step_fn(wl, batch)
    torch.set_num_threads(cands[-1])
    fn()                                   # primitive creation / first-touch, untimed
    best, best_t = cands[0], None
    for c in cands:
        torch.set_num_threads(c)
        fn()
        t0 = time.perf_counter()
        fn()
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best, fn, texels, best_t


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    batch = args.batch or wl['batch']
    cores, fn, texels, _ = calibrate_cpu_threads(wl, args.cpu_batch)
    for _ in range(max(args.warmup, 1)):
        fn()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fn()
    dt = (time.perf_counter() - t0) / args.steps
    val = texels / dt
    sample = 'B=%d of the per-GPU batch %d at %dx%d UV, %s, torch-CPU fp32 restatement of the TF2 path' % (
        args.cpu_batch, batch, wl['uv'], wl['uv'], 'fwd+bwd' if wl['train'] else 'forward')
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': max(args.warmup, 1), 'ms_per_step': dt * 1e3, 'higher_is_better': True, 'scaling': args.scaling,
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args.workload, wl, batch, 1, args.scaling, graph=False),
        'cpu_baseline': {'value': val, 'unit': UNIT, 'cores': cores, 'host_logical_cores': os.cpu_count(),
                         'kind': 'port', 'sample': sample},
        'e2e': {'value': val, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    emit(line)


# ----------------------------------------------------------------------------
# this repo's arm
# ----------------------------------------------------------------------------
def timed(strategy, fn, steps, dev):
    """K steps bracketed by barrier + synchronize, device-timed, max over ranks."""
    strategy.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    strategy.barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if strategy.world > 1:
        torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
    return float(ms) / steps


class TrainRun:
    """One training workload on this rank: model, optimiser, rotating synthetic batches, graphed step."""

    def __init__(self, strategy, wl, batch, global_bs, graph=True, pin=True):
        import models
        import trainvali
        from util import synth
        self.strategy, self.wl, self.batch, self.global_bs = strategy, wl, batch, global_bs
        self.dev = torch.device('cuda', torch.cuda.current_device())
        self.model = models.get_model_class('nlt')(make_config(wl))
        self.model.register_trainable()
        self.opt = trainvali.Adam(learning_rate=1e-3, amsgrad=True)
        uv = wl['uv']
        self.host = [synth.make_batch(batch, uv, uv, seed=1235 + 17 * strategy.rank + i, c_extra=wl['c_extra'],
                                      pin=pin, k_obs=wl['k_obs']) for i in range(2)]
        self.resident = [tuple(t.to(self.dev) if torch.is_tensor(t) else t for t in b) for b in self.host]
        self.graphed = trainvali.GraphedTrainStep(strategy, self.model, self.opt, global_bs) if graph else None
        self.texels = batch * uv * uv * strategy.world

    def step(self, batch, eager=False):
        import trainvali
        if self.graphed is not None and not eager:
            return self.graphed(batch)
        return trainvali.distributed_train_step(self.strategy, self.model, batch, self.opt, self.global_bs)

    def measure_resident(self, steps, warmup):
        import nlt_native as nat
        for i in range(max(warmup, 3)):
            self.step(self.resident[i % 2])
        l0, tc0 = nat.launch_count(), nat.tc_launch_count()
        last = {}

        def fn(i):
            last['out'] = self.step(self.resident[i % 2])
        ms = timed(self.strategy, fn, steps, self.dev)
        self.last_out = last['out']
        launches, tc = nat.launch_count() - l0, nat.tc_launch_count() - tc0
        if self.graphed is not None and self.graphed.graph is not None:
            # replayed kernels are not seen by the library's counter: add the captured ones per replay
            launches += steps * self.graphed.captured_launches
            tc += steps * self.graphed.captured_tc_launches
        return ms, launches, tc

    def measure_e2e(self, steps, uint8=False):
        """pinned host inputs -> H2D each step (copy stream, overlapped with the previous step) -> loss read back.
        uint8: the image tensors of the batch travel as bytes (datasets `uint8_inputs`), normalised on the device."""
        from util import synth
        copy_stream = torch.cuda.Stream()
        state = {}
        host, dev = ([synth.as_uint8(b) for b in self.host] if uint8 else self.host), self.dev

        def prefetch(i):
            with torch.cuda.stream(copy_stream):
                state['next'] = tuple(t.to(dev, non_blocking=True) if torch.is_tensor(t) else t for t in host[i % 2])
                state['ev'] = torch.cuda.Event()
                state['ev'].record(copy_stream)

        def e2e_step(i):
            torch.cuda.current_stream().wait_event(state['ev'])
            cur = state['next']
            prefetch(i + 1)            # overlaps the next step's H2D with this step's compute
            loss, _ = self.step(cur)
            prev = state.get('pending')
            state['pending'] = loss.clone() if self.graphed is not None else loss
            if prev is not None:
                state['loss'] = float(prev)   # D2H read of a step's loss, one step behind the launch front

        prefetch(0)
        for i in range(2):
            e2e_step(i)
        ms = timed(self.strategy, e2e_step, steps, dev)
        torch.cuda.current_stream().wait_event(state['ev'])
        h2d = sum(t.numel() * t.element_size() for t in host[0] if torch.is_tensor(t))
        return ms, h2d

    def per_op(self, rank):
        """roofline leg: per-call CUDA events in a separate eager pass on ONE stream (not the timed value)"""
        import engine
        engine.PROF.enabled = (rank == 0)
        side = engine.USE_SIDE_STREAM
        engine.USE_SIDE_STREAM = False
        try:
            for i in range(2):
                self.step(self.resident[i % 2], eager=True)
        finally:
            engine.USE_SIDE_STREAM = side
        if rank != 0:
            return None
        summ = engine.PROF.summary()
        engine.PROF.enabled = False
        return summ

    def outputs(self):
        """What the last timed step handed its caller: the loss and the tensors the model computed for `to_vis`
        (inputs passed through are left out), plus the parameters after its update and its weight gradients, each
        of the latter flattened in sorted parameter-name order of the Keras layout."""
        loss, to_vis = self.last_out
        params, grads = self.model.export_params(), self.model.export_grads()
        out = {'loss': loss}
        out.update((k, to_vis[k]) for k in ('pred', 'pred_camspc', 'base_camspc', 'gt_camspc'))
        out['params'] = torch.cat([params[k].reshape(-1) for k in sorted(params)])
        out['grads'] = torch.cat([grads[k].reshape(-1) for k in sorted(grads)])
        return out


DUMP_SAMPLE = 1 << 21          # elements kept of a larger output (8 MB in float32); at most 7 outputs are written
DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, arrays):
    """`--dump-outputs`: every array as <out_dir>/<name>.npy, float64 kept and anything else as float32, so that two
    builds can be compared output for output.  An array of more than DUMP_SAMPLE elements is replaced by a fixed
    sample of its flattened elements: one per stride of size // DUMP_SAMPLE, at an offset drawn from a generator
    seeded with 0, in ascending index order (the same positions on every run and every build)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, t in arrays.items():
        a = t.detach()
        a = a if a.dtype == torch.float64 else a.float()
        n = a.numel()
        if n > DUMP_SAMPLE:
            stride = n // DUMP_SAMPLE
            off = torch.randint(stride, (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0))
            a = a.reshape(-1)[(torch.arange(DUMP_SAMPLE) * stride + off).to(a.device)]
        a = a.cpu().numpy()
        total += a.nbytes
        if total > DUMP_LIMIT:
            raise SystemExit('bench.py: --dump-outputs would exceed %d bytes at %s' % (DUMP_LIMIT, name))
        np.save(os.path.join(out_dir, name + '.npy'), a)


def parity_check(run):
    """The bench's own parity gate at the measured shape: the oracle's weights go into the model, one sample of the
    workload runs through both, and `pred_camspc` / the loss must agree to the stated fp32 tolerances
    (max-abs <= 2e-5 against the fp64 oracle, loss relative <= 1e-4) BEFORE anything is timed."""
    from oracle import nlt_oracle as O
    from util import synth
    wl, model = run.wl, run.model
    uv = wl['uv']
    cfg = oracle_cfg(wl)
    params = O.init_params(cfg, c_query=5 + wl['c_extra'], seed=7, dtype=torch.float64)
    bt = synth.make_batch(1, uv, uv, seed=4321, c_extra=wl['c_extra'], k_obs=wl['k_obs'])
    model.build(5 + wl['c_extra'], 3)
    saved = model.flat_params.clone()
    model.load_params(params)
    t0 = time.perf_counter()
    with torch.no_grad():
        p64, g64, _, _ = O.model_call(params, cfg, tuple(t.double() if torch.is_tensor(t) else t for t in bt), 'train')
        l64 = float(O.l2_loss(g64, p64, keep_batch=True)[0])
    t_oracle = time.perf_counter() - t0
    pred, gt, kw, _ = model(bt, mode='vali')
    kw['keep_batch'] = True
    loss = float(model.compute_loss(pred, gt, **kw)[0])
    err = float((pred.double().cpu() - p64).abs().max())
    gerr = float((gt.double().cpu() - g64).abs().max())
    model.flat_params.copy_(saved)
    rel = abs(loss - l64) / max(abs(l64), 1e-30)
    res = {'shape': 'B=1 at %dx%d, %d query channels, K=%d' % (uv, uv, 5 + wl['c_extra'], wl['k_obs']),
           'pred_camspc_max_abs': err, 'gt_camspc_max_abs': gerr, 'loss_rel': rel, 'tol_pred': 2e-5, 'tol_loss': 1e-4,
           'oracle': 'fp64 torch-CPU restatement (oracle/nlt_oracle.py), %.1f s' % t_oracle,
           'ok': bool(err <= 2e-5 and gerr <= 2e-5 and rel <= 1e-4)}
    if not res['ok']:
        raise SystemExit('bench.py: parity gate failed at the measured shape: %s' % json.dumps(res))
    return res


def measure_tf32_peak(dev):
    """Dense TF32 tensor-core peak of this box (cuBLAS through torch.matmul, 8192^3, best of 5): the FLOP roofline's
    denominator.  The 3xTF32 kernels issue three tensor-core products per algorithmic product."""
    n = 8192
    a = torch.randn(n, n, device=dev)
    b = torch.randn(n, n, device=dev)
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        best = None
        for _ in range(6):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            best = ms if best is None or ms < best else best
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    del a, b
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12


def forward_record(strategy, wl, batch, steps, warmup, dump_dir=None):
    """cfg1: forward only (mode 'test') through the cached observation features, device-resident and end to end."""
    import models
    import nlt_native as nat
    import nlt_test
    from util import synth
    dev = torch.device('cuda', torch.cuda.current_device())
    uv = wl['uv']
    model = models.get_model_class('nlt')(make_config(wl))
    model.register_trainable()
    model.build(5 + wl['c_extra'], 3)
    host = [synth.make_batch(batch, uv, uv, seed=99 + i, c_extra=wl['c_extra'], pin=True) for i in range(2)]
    resident = [tuple(t.to(dev) if torch.is_tensor(t) else t for t in b) for b in host]
    feat = nlt_test.extract_feat(model, [resident[0]], 1)
    for i in range(max(warmup, 3)):
        model.call(resident[i % 2], 'test', obs_override=feat)
    l0 = nat.launch_count()
    last = {}

    def fwd(i):
        last['out'] = model.call(resident[i % 2], 'test', obs_override=feat)
    ms = timed(strategy, fwd, steps, dev)
    launches = nat.launch_count() - l0
    if dump_dir is not None and strategy.rank == 0:
        pred_c, _, _, to_vis = last['out']
        dump_outputs(dump_dir, {'pred_camspc': pred_c, 'pred': to_vis['pred'], 'base_camspc': to_vis['base_camspc']})

    def e2e(i):
        b = tuple(t.to(dev, non_blocking=True) if torch.is_tensor(t) else t for t in host[i % 2])
        pred = model.call(b, 'test', obs_override=feat)[0]
        e2e.last = pred[0, 0, 0].cpu()        # D2H read of a piece of the result
    for i in range(2):
        e2e(i)
    ms_e2e = timed(strategy, e2e, steps, dev)
    texels = batch * uv * uv
    peak_gbs, _, _ = measured_peaks()
    return {'ms_per_step': ms, 'value': texels / (ms * 1e-3), 'e2e_ms_per_step': ms_e2e,
            'e2e_value': texels / (ms_e2e * 1e-3), 'gpu_launches': launches,
            'hbm_frac': wl['bytes'][0] * texels / (ms * 1e-3) / 1e9 / peak_gbs,
            'alg_bytes_per_texel': wl['bytes'][0]}


def sub_record(args):
    """`--sub NAME[:batch]`: one short measurement of another workload in THIS process (the parent isolates every
    sub-record in its own process so that an out-of-memory or an illegal address there cannot take the headline
    down); prints a compact JSON record."""
    import trainvali
    name, _, b = args.sub.partition(':')
    wl = WORKLOADS[name]
    batch = int(b) if b else wl['batch']
    strategy = trainvali.Strategy()
    peak_gbs, _, _ = measured_peaks()
    rec = {'workload': name, 'batch_per_gpu': batch, 'uv': wl['uv'], 'query_channels': 5 + wl['c_extra'],
           'observations': wl['k_obs'], 'kernel': wl['kernel'], 'depth': wl['depth'],
           'mode': 'fwd+L2+bwd+AMSGrad' if wl['train'] else 'forward only (obs_override)'}
    if not wl['train']:
        rec.update(forward_record(strategy, wl, batch, args.steps, args.warmup))
    else:
        run = TrainRun(strategy, wl, batch, batch * strategy.world)
        ms, launches, tc = run.measure_resident(args.steps, args.warmup)
        ms_e2e, h2d = run.measure_e2e(args.steps)
        rec.update({'ms_per_step': ms, 'value': run.texels / (ms * 1e-3), 'e2e_ms_per_step': ms_e2e,
                    'e2e_value': run.texels / (ms_e2e * 1e-3), 'h2d_bytes_per_step': h2d,
                    'gpu_launches_per_step': launches / args.steps, 'tcgen05_launches_per_step': tc / args.steps,
                    'hbm_frac': wl['bytes'][1] * run.texels / (ms * 1e-3) / 1e9 / peak_gbs,
                    'alg_bytes_per_texel': wl['bytes'][1],
                    'peak_mem_GB': torch.cuda.max_memory_allocated() / 1e9})
    emit(rec)


def collect_extra(args):
    """Sub-records of the default N = 1 run, each in its own process (see sub_record)."""
    out = []
    subs = ['cfg4:1', 'cfg4:32', 'cfg2:8', 'cfg2:1', 'cfg4k3:8', 'cfg1:1', 'cfg3:16']
    for sub in subs:
        name = sub.split(':')[0]
        if name == args.workload and sub.endswith(':%d' % (args.batch or WORKLOADS[name]['batch'])):
            continue
        cmd = [sys.executable, os.path.abspath(__file__), '--sub', sub, '--steps', str(min(args.steps, 5)),
               '--warmup', '3']
        try:
            r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=args.sub_timeout)
            lines = [ln for ln in r.stdout.decode().splitlines() if ln.startswith('{')]
            if r.returncode == 0 and lines:
                out.append(json.loads(lines[-1]))
            else:
                out.append({'workload': name, 'sub': sub, 'error': (r.stderr.decode().strip().splitlines() or ['rc %d' % r.returncode])[-1][:300]})
        except subprocess.TimeoutExpired:
            out.append({'workload': name, 'sub': sub, 'error': 'timeout after %d s' % args.sub_timeout})
    return out


def run_b200(args):
    import trainvali
    import engine
    wl = WORKLOADS[args.workload]
    strategy = trainvali.Strategy()
    world, rank = strategy.world, strategy.rank
    dev = torch.device('cuda', torch.cuda.current_device())
    if args.scaling == 'strong':
        gb = args.global_batch or 32
        batch = max(gb // world, 1)
    else:
        batch = args.batch or wl['batch']
    global_bs = batch * world

    if not wl['train']:
        rec = forward_record(strategy, wl, batch, args.steps, args.warmup, args.dump_outputs)
        if rank == 0:
            emit({'metric': 'UV texels/sec fwd', 'value': rec['value'], 'unit': UNIT, 'n_gpus': world,
                  'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': rec['ms_per_step'],
                  'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None, 'dtype': 'f32',
                  'data': 'synthetic', 'config': workload_config(args.workload, wl, batch, world, args.scaling, False),
                  'e2e': {'value': rec['e2e_value'], 'unit': UNIT, 'ms_per_step': rec['e2e_ms_per_step']},
                  'gpu_launches': rec['gpu_launches'], 'roofline': {'bound': 'hbm', 'frac': rec['hbm_frac']}})
        return

    run = TrainRun(strategy, wl, batch, global_bs, graph=not args.no_graph)
    parity = parity_check(run) if rank == 0 and not args.no_parity else None

    # ---- device-resident arm ("value") ----
    sampler = ClockSampler(torch.cuda.current_device())
    for i in range(max(args.warmup, 3)):
        run.step(run.resident[i % 2])
    if rank == 0:
        sampler.start()
    ms_step, launches, tc_launches = run.measure_resident(args.steps, 0)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, run.outputs())

    # ---- end-to-end arm ----
    ms_e2e, h2d_bytes = run.measure_e2e(args.steps)
    ms_e2e_u8, h2d_bytes_u8 = run.measure_e2e(args.steps, uint8=True)

    # ---- roofline leg ----
    summ = run.per_op(rank)       # every rank runs these steps (they contain the gradient all-reduce)
    roof = None
    if rank == 0:
        total_ms = sum(v['ms'] for v in summ.values())
        top_label, top = max(summ.items(), key=lambda kv: kv[1]['ms'])
        peak_gbs, peak_bf16, how = measured_peaks()
        tf32_peak = measure_tf32_peak(dev)
        ach = top['bytes'] / (top['ms'] * 1e-3) / 1e9
        texels_rank = batch * wl['uv'] * wl['uv']
        step_bytes = wl['bytes'][1] * texels_rank
        step_flops = 3.0 * wl['flop_fwd'] * texels_rank
        roof = {
            'bound': 'hbm', 'achieved': ach, 'peak': peak_gbs, 'unit': 'GB/s', 'frac': ach / peak_gbs,
            'traffic': ncu_traffic(top_label), 'peak_source': how + ' copy bandwidth (MEASURED_PEAKS.json hbm_gbs)'
            if how == 'measured' else 'fallback 6.65 TB/s (B200_PROFILING.md)',
            'kernel': top_label, 'kernel_launches_per_step': top['launches'] / 2,
            'kernel_ms_per_launch': top['ms'] / top['launches'],
            'kernel_alg_bytes_per_launch': top['bytes'] / top['launches'],
            'kernel_share_of_step': top['ms'] / total_ms,
            'step': {'alg_bytes': step_bytes, 'alg_bytes_per_texel': wl['bytes'][1],
                     'achieved_GBps': step_bytes / (ms_step * 1e-3) / 1e9,
                     'hbm_frac': step_bytes / (ms_step * 1e-3) / 1e9 / peak_gbs,
                     'conv_granular_bytes': sum(v['bytes'] for v in summ.values()) / 2,
                     'alg_flops': step_flops,
                     'tf32_peak_tflops_measured': tf32_peak,
                     'flop_frac_of_tf32_peak': step_flops / (ms_step * 1e-3) / 1e12 / tf32_peak,
                     'flop_note': 'algorithmic conv FLOPs (fwd+bwd = 3 x fwd); the tcgen05 kernels spend 3 TF32 '
                                  'products per algorithmic product (3xTF32 split), the fp32 kernels none'},
            'per_op_sum_ms': total_ms / 2,
            'top5': sorted(((k, round(v['ms'] / 2, 4)) for k, v in summ.items()), key=lambda kv: -kv[1])[:5],
        }
        if args.profile_out:
            rows = sorted(({'op': k, 'ms_per_step': v['ms'] / 2, 'launches_per_step': v['launches'] / 2,
                            'alg_MB_per_step': v['bytes'] / 2 / 1e6,
                            'GBps': v['bytes'] / (v['ms'] * 1e-3) / 1e9} for k, v in summ.items()),
                          key=lambda r: -r['ms_per_step'])
            json.dump({'ms_step': ms_step, 'sum_ms': total_ms / 2, 'rows': rows}, open(args.profile_out, 'w'), indent=1)

    run_graph_full = run.graphed is not None and run.graphed.full_step_in_graph
    # ---- strong-scaling sub-record (N > 1): cfg4's FIXED global batch 32 ----
    strong = None
    if world > 1 and args.scaling == 'weak' and not args.no_extra and 32 % world == 0:
        del run
        torch.cuda.empty_cache()
        srun = TrainRun(strategy, wl, 32 // world, 32)
        sms, _, _ = srun.measure_resident(min(args.steps, 10), 3)
        strong = {'scaling': 'strong', 'global_batch': 32, 'batch_per_gpu': 32 // world, 'ms_per_step': sms,
                  'value': 32 * wl['uv'] * wl['uv'] / (sms * 1e-3), 'n_gpus': world,
                  'collectives_in_graph': bool(srun.graphed.full_step_in_graph)}
        del srun

    # ---- CPU baseline (rank 0, N=1 only): bounded sample of the same workload ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores, fn, texels, _ = calibrate_cpu_threads(wl, args.cpu_batch)
        t0 = time.perf_counter()
        n = 2
        for _ in range(n):
            fn()
        dt = (time.perf_counter() - t0) / n
        cpu = {'value': texels / dt, 'unit': UNIT, 'cores': cores, 'host_logical_cores': os.cpu_count(),
               'kind': 'port',
               'sample': 'B=%d of the B=%d step at %dx%d UV (%d query channels), fwd+bwd, thread count calibrated at '
                         'this size, %d timed passes, torch-CPU fp32 restatement of the TF2 path (TensorFlow is not '
                         'installable offline)' % (args.cpu_batch, batch, wl['uv'], wl['uv'], 5 + wl['c_extra'], n)}

    extra = None
    if rank == 0 and world == 1 and not args.no_extra:
        torch.cuda.empty_cache()
        extra = collect_extra(args)

    if rank == 0:
        texels_step = batch * wl['uv'] * wl['uv'] * world
        line = {
            'metric': METRIC, 'value': texels_step / (ms_step * 1e-3), 'unit': UNIT, 'n_gpus': world,
            'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': ms_step, 'higher_is_better': True,
            'scaling': args.scaling, 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': workload_config(args.workload, wl, batch, world, args.scaling, not args.no_graph),
            'e2e': {'value': texels_step / (ms_e2e * 1e-3), 'unit': UNIT, 'ms_per_step': ms_e2e,
                    'h2d_bytes_per_step': h2d_bytes, 'd2h_bytes_per_step': 4,
                    'note': 'float32 host buffers (the reference tuple\'s dtypes) copied H2D every step on a copy '
                            'stream; the loss (4 bytes) is the result read back -- a train step returns nothing else',
                    'uint8_inputs': {'value': texels_step / (ms_e2e_u8 * 1e-3), 'unit': UNIT, 'ms_per_step': ms_e2e_u8,
                                     'h2d_bytes_per_step': h2d_bytes_u8,
                                     'note': 'same call with the image tensors as uint8 PNG samples (datasets '
                                             'uint8_inputs = True; v / 255 on the device, bit-identical results); the '
                                             'float32 number above is bounded by PCIe (h2d bytes / step time)'}},
            'gpu_launches': launches, 'tcgen05_launches': tc_launches,
            'whole_step_in_cuda_graph': bool(run_graph_full), 'clocks': clocks, 'parity': parity,
            'roofline': roof, 'cpu_baseline': cpu,
        }
        if strong is not None:
            line['strong_scaling'] = strong
        if extra is not None:
            line['extra'] = extra
        emit(line)
    if world > 1:
        torch.distributed.destroy_process_group()


def ncu_traffic(label):
    """DRAM bytes per launch of the dominant kernel, from the committed ncu --set full capture
    (profiles/ncu_traffic.json); None when that kernel has not been captured."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'ncu_traffic.json')) as f:
            ent = json.load(f).get(label)
        return float(ent['dram_bytes_per_launch']) if ent else None
    except (OSError, ValueError, KeyError):
        return None


_JSON_OUT = None


def _guard_stdout():
    """Keep stdout to the ONE JSON line of the contract: native libraries write banners to fd 1
    (NCCL prints its version there on the first communicator), so fd 1 is pointed at stderr and the
    result line goes to a private duplicate of the original stdout."""
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), 'w')
    os.dup2(2, 1)


def emit(line):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + '\n')
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='cfg4', choices=sorted(WORKLOADS))
    ap.add_argument('--batch', type=int, default=None, help='per-GPU batch (default: the workload\'s)')
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'],
                    help='N > 1: weak = per-GPU batch fixed; strong = global batch fixed (--global-batch, default 32)')
    ap.add_argument('--global-batch', dest='global_batch', type=int, default=None)
    ap.add_argument('--cpu-batch', dest='cpu_batch', type=int, default=1)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extra', action='store_true', help='skip the sub-records of the other workloads')
    ap.add_argument('--no-parity', action='store_true', help='skip the in-bench parity gate')
    ap.add_argument('--no-graph', dest='no_graph', action='store_true', help='launch kernels eagerly (no CUDA graph)')
    ap.add_argument('--profile-out', dest='profile_out', default=None, help='write the per-op device-time table here')
    ap.add_argument('--dump-outputs', dest='dump_outputs', default=None, metavar='DIR',
                    help='after the timed steps, write what the last one computed as DIR/<name>.npy (rank 0)')
    ap.add_argument('--sub', default=None, help=argparse.SUPPRESS)
    ap.add_argument('--sub-timeout', dest='sub_timeout', type=int, default=240, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'b200' or args.sub):
        ap.error('--dump-outputs writes the outputs of the B200 path (--impl b200)')
    _guard_stdout()
    if args.impl == 'reference':
        run_reference(args)
        return
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device (the B200 path has no CPU fallback); '
                         'use --impl reference for the CPU arm')
    if args.sub:
        sub_record(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
