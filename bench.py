"""bench.py -- headline benchmark of the general_cf training hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload simgcl-amazon] [--dump-outputs DIR]

The GPU arm times each training-step loop over K steps after W warm-up steps; the value is the median of five such passes
of the resident-batch loop.  ``--dump-outputs DIR`` writes what the last step of the last of those passes returned (see
``outputs_of_step``) once the timed steps are done.  The same arguments give the same graph, weights and batches; the
backward adds with floating-point atomics, so two runs agree to rounding (amplified in the parameters by Adam's division),
not bit for bit.

One "step" = one iteration of trainer/trainer.py:63-68 (zero_grad, cal_loss, backward, Adam step) at
B = 4096 on BASELINE.json configs[1]: SimGCL, d = 64, L = 3, tau = 0.2, on a synthetic graph with the
reference's amazon shape (|U| = 76 469, |I| = 83 761, nnz = 2 x 966 680; synth_graphs.py).
Prints ONE JSON line (contract in the task statement):
  value      steps/s with the batch indices already resident in HBM (CUDA events, max over ranks)
  e2e        steps/s through the plugin surface from pinned HOST index buffers, with the H2D copy of
             the batch and the D2H reads of loss / loss terms (loss.item(), float(v)) in the timed region
  roofline   the propagation SpMM kernel (HBM-bound): algorithmic bytes / live CUDA-event time
  cpu_baseline  the oracle port of the reference's CPU path, timed on this box's host cores
``--impl reference`` times that CPU path alone (rank 0 only under torchrun).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

WORKLOADS = {
    # name: (model, graph, model hyper-parameters)   -- BASELINE.json configs
    'simgcl-amazon': ('simgcl', 'amazon', dict(layer_num=3, embedding_size=64, temperature=0.2, eps=0.9, cl_weight=1.0e-2,
                                               reg_weight=1.0e-6, keep_rate=1.0)),
    'lightgcn-gowalla': ('lightgcn', 'gowalla', dict(layer_num=3, embedding_size=64, reg_weight=1.0e-8, keep_rate=0.5)),
    'sgl-yelp': ('sgl', 'yelp', dict(layer_num=3, embedding_size=64, temperature=0.2, cl_weight=1.0, reg_weight=1.0e-5,
                                     keep_rate=0.5, augmentation='edge_drop')),
    # BASELINE.json configs[3]: row-sharded over the GPUs (bench_rowshard.py); the whole 10 M x 2 M / 300 M-edge graph at any N
    'lightgcn-xl': ('lightgcn', 'synthetic-xl', dict(layer_num=3, embedding_size=128, reg_weight=1.0e-8, keep_rate=1.0)),
    'lightgcn-xl-8th': ('lightgcn', 'synthetic-xl-8th', dict(layer_num=3, embedding_size=128, reg_weight=1.0e-8, keep_rate=1.0)),
    'ncl-amazon': ('ncl', 'amazon', dict(layer_num=3, embedding_size=64, high_order=2, reg_weight=1.0e-7, proto_weight=1.0e-4,
                                         struct_weight=1.0e-3, temperature=0.1, epoch_period=3, cluster_num=50, keep_rate=1.0)),
    'lightgcl-gowalla': ('lightgcl', 'gowalla', dict(layer_num=2, embedding_size=64, dropout=0.0, cl_weight=0.1, reg_weight=1.0e-9, temp=0.1, svd_q=5)),
    'directau-gowalla': ('directau', 'gowalla', dict(layer_num=2, embedding_size=64, gamma=2.0)),
    'hccf-amazon': ('hccf', 'amazon', dict(layer_num=2, embedding_size=64, reg_weight=1.0e-7, cl_weight=1.0, temperature=0.1,
                                           keep_rate=0.5, mult=1.0, hyper_num=128, leaky=0.5)),
}
BATCH = 4096


def rank_world():
    return int(os.environ.get('RANK', 0)), int(os.environ.get('LOCAL_RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))


def graph_arrays(name):
    from synth_graphs import named_graph
    cache = os.path.join('/tmp', f'sslrec_b200_graph_{name}.npz')
    if os.path.exists(cache):
        z = np.load(cache)
        return z['rows'], z['cols'], int(z['n_user']), int(z['n_item'])
    rows, cols, n_user, n_item = named_graph(name, seed=2023)
    try:
        np.savez(cache + f'.{os.getpid()}.npz', rows=rows, cols=cols, n_user=n_user, n_item=n_item)
        os.replace(cache + f'.{os.getpid()}.npz', cache)
    except OSError:
        pass
    return rows, cols, n_user, n_item


def make_batches(rows, cols, n_item, count, seed=2023):
    """``count`` batches of (ancs, poss, negs): B uniform training edges + uniform negatives (the
    DataLoader's shuffle + sample_negs draw, pre-materialised so the timed region holds no Python sampling)."""
    rs = np.random.RandomState(seed)
    out = []
    for _ in range(count):
        pick = rs.randint(0, len(rows), size=BATCH)
        out.append(np.stack([rows[pick], cols[pick], rs.randint(0, n_item, size=BATCH)]).astype(np.int64))
    return out


DUMP_LIMIT = 64 * 10 ** 6      # bytes of --dump-outputs in all
DUMP_GRAD_ROWS = 4096          # gradient rows sampled per parameter


def outputs_of_step(model, loss, parts):
    """Host copies of what one training step hands its caller: the loss, every loss term, the parameters after the optimizer
    step (in full while they fit 3/4 of DUMP_LIMIT, else a seeded sample of rows) and a seeded sample of DUMP_GRAD_ROWS rows of
    each gradient.  The row samples depend only on the parameter shapes, so two runs with the same arguments pick the same rows."""
    out = {'loss': loss.detach().float().cpu().numpy()}
    for k, v in parts.items():
        out['part_' + k] = torch.as_tensor(v).detach().float().cpu().numpy()
    named = [(n, p) for n, p in model.named_parameters()]
    full = sum(p.numel() for _, p in named) * 4 <= DUMP_LIMIT * 3 // 4
    for i, (n, p) in enumerate(named):
        x = p.detach().float()
        if not full and x.dim() > 0 and x.shape[0] > 1:
            rows = max(1, x.shape[0] * (DUMP_LIMIT * 3 // 4) // (4 * sum(q.numel() for _, q in named)))
            x = x[torch.from_numpy(np.sort(np.random.RandomState(i).choice(x.shape[0], min(rows, x.shape[0]), replace=False))).to(x.device)]
        out['param_' + n] = x.cpu().numpy()
        if p.grad is not None:
            g = p.grad.detach().float()
            if g.dim() > 0 and g.shape[0] > DUMP_GRAD_ROWS:
                g = g[torch.from_numpy(np.sort(np.random.RandomState(1000 + i).choice(g.shape[0], DUMP_GRAD_ROWS, replace=False))).to(g.device)]
            out['grad_' + n] = g.cpu().numpy()
    return out


def write_outputs(path, arrays):
    """``path/<name>.npy`` for every array (float32; at most DUMP_LIMIT bytes in all)."""
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise RuntimeError(f'--dump-outputs: {total} bytes exceed the {DUMP_LIMIT} byte limit')
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k.replace('/', '_') + '.npy'), np.ascontiguousarray(a, dtype=np.float32))


class ClockSampler:
    """SM clock / throttle reasons read through NVML from the benchmarking thread itself WHILE the GPU
    works through the enqueued steps (a polling nvidia-smi subprocess perturbed the timed region by
    25 % in round 1, so no subprocess, no sampler thread)."""
    REASONS = {0x8: 'hw_slowdown', 0x40: 'hw_thermal_slowdown', 0x20: 'sw_thermal_slowdown', 0x4: 'sw_power_cap',
               0x80: 'hw_power_brake_slowdown'}

    def __init__(self, gpu_index):
        self.sm, self.mx, self.power, self.reasons, self.h = [], None, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:      # noqa: BLE001
            self.err = repr(e)

    def sample(self):
        if self.h is None:
            return
        nv = self.nv
        try:
            self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
            self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            get = getattr(nv, 'nvmlDeviceGetCurrentClocksEventReasons', None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
            bits = int(get(self.h))
            for bit, name in self.REASONS.items():
                if bits & bit:
                    self.reasons.add(name)
        except Exception as e:      # noqa: BLE001
            self.err = repr(e)

    def drain(self, event, period_s=0.02):
        """Sample until ``event`` (recorded after the last timed step) has completed."""
        while not event.query():
            self.sample()
            time.sleep(period_s)

    def result(self):
        if self.h is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvml unavailable: ' + getattr(self, 'err', '?')]}
        return {'sm_mhz': float(np.median(self.sm)) if self.sm else None, 'sm_max_mhz': self.mx, 'reasons': sorted(self.reasons),
                'samples': len(self.sm), 'power_w_max': max(self.power) if self.power else None}


def ncu_traffic(kernel, key):
    """DRAM bytes per launch from the committed ncu capture of this workload (profiles/traffic.json), else None."""
    p = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(p):
        return json.load(open(p)).get(kernel, {}).get(key)
    return None


def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        return json.load(open(p)), 'measured'
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0}, 'fallback'


# --------------------------------------------------------------------------------------------------
# the CPU arm: oracle port of the reference path (oracle/cf_oracle.CpuTrainer)
# --------------------------------------------------------------------------------------------------

def usable_cpus():
    """Host cores this process may actually burn: the affinity mask capped by the cgroup CPU quota (cpu.max)."""
    n = len(os.sched_getaffinity(0))
    try:
        quota, period = open('/sys/fs/cgroup/cpu.max').read().split()
        if quota != 'max':
            n = max(1, min(n, int(math.ceil(int(quota) / int(period)))))
    except (OSError, ValueError):
        pass
    return n


def cpu_steps(model, hp, rows, cols, n_user, n_item, batches, budget_s, max_steps, warmup=1, csr=False, threads=None):
    """csr=True: the "tuned CPU" variant of SURVEY.md 8(d) (adjacency converted with to_sparse_csr(), everything else the
    reference's path); ``threads`` skips the thread-count calibration."""
    from oracle import cf_oracle as O
    adj = O.normalized_adjacency(rows, cols, n_user, n_item)
    adj.reference_layout = True                      # the reference's column-sorted COO (data_handler_general_cf.py:69-72)
    tr = O.CpuTrainer(model, adj, hp['embedding_size'], dict(hp, lr=1e-3), csr=csr)
    tb = [tuple(torch.from_numpy(b[i]) for i in range(3)) for b in batches]
    t_start = time.perf_counter()
    # all usable host threads (affinity capped by the cgroup quota), unless 32 are faster (torch's sparse COO addmm stops scaling early): one
    # untimed step per candidate doubles as the warm-up
    cands = [threads] if threads else sorted({usable_cpus(), min(usable_cpus(), 32)}, reverse=True)
    best, threads = None, cands[0]
    for c in cands:
        torch.set_num_threads(c)
        t0 = time.perf_counter()
        tr.step(tb[0])
        dt = time.perf_counter() - t0
        if best is None or dt < best:
            best, threads = dt, c
    torch.set_num_threads(threads)
    times = []
    for i in range(max_steps):
        t0 = time.perf_counter()
        tr.step(tb[(warmup + i) % len(tb)])
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_start > budget_s:
            break
    return times, threads


def reference_available():
    """The unmodified reference, vendored to oracle/_ref by oracle/vendor_ref.py (build() runs the recipe)."""
    try:
        from oracle import vendor_ref
        return vendor_ref.available() or os.path.isdir(vendor_ref.REF)
    except Exception:      # noqa: BLE001
        return False


def reference_steps(model, hp, rows, cols, n_user, n_item, batches, budget_s, max_steps, warmup=1, csr=False, threads=None):
    """Seconds per step of the reference's CPU path on this box's host cores: the UNMODIFIED reference (oracle/_ref,
    kind "reference") when it is there, else the oracle port (kind "port")."""
    if reference_available() and model in ('lightgcn', 'simgcl', 'sgl', 'ncl', 'hccf', 'directau', 'lightgcl'):
        from oracle import ref_runner
        cands = [threads] if threads else sorted({usable_cpus(), min(usable_cpus(), 32)}, reverse=True)
        times, used = ref_runner.time_steps(model, rows, cols, n_user, n_item, hp, batches, cands, budget_s, max_steps, warmup=warmup, csr=csr)
        return times, used, 'reference'
    times, used = cpu_steps(model, hp, rows, cols, n_user, n_item, batches, budget_s, max_steps, warmup=warmup, csr=csr, threads=threads)
    return times, used, 'port'


def run_reference(args):
    """The reference arm: no GPU work and nothing of sslrec_b200 is imported in this process."""
    rank, _, world = rank_world()
    if rank != 0:
        return
    model, graph, hp = WORKLOADS[args.workload]
    if not reference_available() and model not in ('lightgcn', 'simgcl', 'sgl', 'directau'):
        print(json.dumps({'impl': 'reference', 'unavailable': f'oracle/_ref is absent and oracle.CpuTrainer has no whole-step driver for {model}'}))
        return
    if graph.startswith('synthetic-xl'):
        print(json.dumps({'impl': 'reference', 'unavailable': 'config 4 (600 M stored entries) does not fit the bounded CPU sample; see cpu_baseline of lightgcn-xl-8th'}))
        return
    rows, cols, n_user, n_item = graph_arrays(graph)
    batches = make_batches(rows, cols, n_item, max(2, min(args.steps + args.warmup, 8)))
    times, threads, kind = reference_steps(model, hp, rows, cols, n_user, n_item, batches, budget_s=args.cpu_budget, max_steps=args.steps,
                                           warmup=max(1, min(args.warmup, 2)), csr=args.cpu_csr)
    ms = 1e3 * float(np.median(times))
    val = 1e3 / ms
    what = ('the unmodified reference (oracle/_ref: build_data_handler, build_model, Trainer.create_optimizer, the trainer.py:63-68 loop)'
            if kind == 'reference' else 'oracle port of the reference CPU path')
    sample = (f'{len(times)} of {args.steps} full training steps executed inside the {args.cpu_budget:.0f} s budget (median step time); '
              f'{what}, torch {torch.__version__} sparse {"CSR" if args.cpu_csr else "COO"} spmm + dense InfoNCE, {threads} threads')
    print(json.dumps({
        'impl': 'reference', 'metric': 'train_steps_per_sec', 'value': val, 'unit': 'steps/s', 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True,
        'scaling': scaling_label(args.parallel, args.workload, n_user, n_item, world),
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args.workload, n_user, n_item, len(rows), world, parallel_mode(args.parallel, args.workload, n_user, n_item, world)),
        'cpu_baseline': {'value': val, 'unit': 'steps/s', 'cores': threads, 'kind': kind, 'sample': sample},
        'e2e': {'value': val, 'unit': 'steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'sslrec_b200_imported': 'sslrec_b200' in sys.modules,
    }))


def cpu_baseline_subprocess(workload, steps, budget_s, csr=False):
    """The cpu_baseline leg of the GPU arm: the reference arm in its own process (the reference's config is a module-level
    singleton and its harness shims torch.Tensor.cuda -- neither belongs in the process that measures the GPU)."""
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--workload', workload, '--steps', str(steps), '--warmup', '1',
           '--cpu-budget', str(budget_s)] + (['--cpu-csr'] if csr else [])
    env = {k: v for k, v in os.environ.items() if k not in ('RANK', 'LOCAL_RANK', 'WORLD_SIZE')}
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=budget_s * 4 + 120, env=env)
    for line in reversed(r.stdout.strip().splitlines()):
        if line.startswith('{'):
            return json.loads(line)
    raise RuntimeError('reference arm printed no JSON line: ' + r.stderr[-400:])


class Watchdog:
    """If the optional row-shard leg wedges (a rank died inside a collective), still deliver the bench line: after
    ``deadline_s`` the fallback is printed by rank 0 and every rank leaves with exit code 0."""

    def __init__(self, deadline_s, fallback):
        self.timer = threading.Timer(deadline_s, self._fire)
        self.timer.daemon = True
        self.fallback = fallback
        self.timer.start()

    def _fire(self):
        try:
            line = self.fallback()
            if line is not None:
                print(line, flush=True)
        finally:
            os._exit(0)

    def cancel(self):
        self.timer.cancel()


def n_views(model):
    return 3 if model in ('simgcl', 'sgl') else 1


def parallel_mode(requested, name, n_user, n_item, world):
    """How N > 1 GPUs are used (sslrec_b200/parallel.py).  'dp': every rank steps on its own batch of B and the
    parameter gradients are averaged (one all-reduce) -- the batches are the sharded unit, weak scaling.  'shard': one
    batch of B, table rows sharded (InfoNCE always, propagation when the table is >= 1 GiB) -- strong scaling.
    'auto' row-shards when the layer tensors are HBM-scale (BASELINE.json config 4) and data-parallels otherwise."""
    if world == 1:
        return 'single'
    if requested != 'auto':
        return requested
    model, _, hp = WORKLOADS[name]
    return 'shard' if (n_user + n_item) * n_views(model) * hp['embedding_size'] * 4 >= (1 << 30) else 'dp'


def scaling_label(requested, name, n_user, n_item, world):
    """'weak' when N > 1 GPUs would each take their own batch (the N = 1 line carries the same label so that the driver's
    1 -> N series is labelled consistently), 'strong' when one batch is sharded."""
    return 'weak' if parallel_mode(requested, name, n_user, n_item, max(world, 2)) == 'dp' else 'strong'


def workload_config(name, n_user, n_item, n_edge, world, mode='single'):
    model, graph, hp = WORKLOADS[name]
    shard_prop = (n_user + n_item) * n_views(model) * hp['embedding_size'] * 4 >= (1 << 30)
    par = {'single': 'single GPU',
           'dp': f'dp{world}: one batch of {BATCH} per GPU per step, parameter gradients averaged by one NCCL all-reduce before Adam '
                 f'(= one reference step at batch_size {world * BATCH}); a "step" in value/e2e is one {BATCH}-sample batch',
           'shard': f'x{world}: one batch of {BATCH} per step; InfoNCE table rows sharded; propagation '
                    + ('row-sharded (all-gather per layer)' if shard_prop else 'replicated (table < 1 GiB)')}[mode]
    return {'workload': f'{model} training step on synthetic {graph}-shaped graph', 'model_name': model, 'graph': graph,
            'n_user': n_user, 'n_item': n_item, 'nnz': 2 * n_edge, 'batch': BATCH, 'global_batch': BATCH * (world if mode == 'dp' else 1),
            'dim': hp['embedding_size'], 'layers': hp['layer_num'], 'temperature': hp.get('temperature'), 'parallelism': par,
            'propagation': 'one prop_kernel launch per layer and direction (2L per step; a layer needs every row of the previous one), layer sum and '
                           'augmentation fused into the launches',
            'l2': 'no explicit flush: each step touches > 1 GB (3-view activations, gradient sinks, split partials) >> 126 MB L2'}


# --------------------------------------------------------------------------------------------------
# the GPU arm
# --------------------------------------------------------------------------------------------------

def run_ours(args):
    rank, local_rank, world = rank_world()
    import scipy.sparse as sp
    import sslrec_b200
    from sslrec_b200 import _lib, engine
    from sslrec_b200.config import default_config, load_config
    from sslrec_b200.data_handler import DataHandlerGeneralCF
    from sslrec_b200.optim import FusedAdam

    torch.cuda.set_device(local_rank)
    torch.set_num_threads(min(4, torch.get_num_threads()))      # the GPU arm has no CPU math; idle OpenMP spinners only eat the cgroup quota
    dev = torch.device('cuda', local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=dev)
    model_name, graph, hp = WORKLOADS[args.workload]
    rows, cols, n_user, n_item = graph_arrays(graph)
    cfg = default_config(model_name, **hp)
    cfg['train']['batch_size'] = BATCH
    if model_name == 'ncl':
        cfg['train']['loss'] = 'pairwise_with_epoch_flag'
    load_config(base=cfg, device=str(dev))
    trn = sp.coo_matrix((np.ones(len(rows), dtype=np.float32), (rows, cols)), shape=(n_user, n_item))
    dh = DataHandlerGeneralCF(trn)
    dh.load_data()
    import importlib
    mod = importlib.import_module('sslrec_b200.general_cf.' + model_name)
    cls = [getattr(mod, a) for a in dir(mod) if a.lower() == model_name][0]
    torch.manual_seed(2023)
    model = cls(dh)
    mode = parallel_mode(args.parallel, args.workload, n_user, n_item, world)
    sync = None
    if mode == 'shard':
        from sslrec_b200.parallel import RowShard
        model.comm = RowShard(dist, rank, world, n_user + n_item, dim=hp['embedding_size'], views=n_views(model_name))
    elif mode == 'dp':
        from sslrec_b200.parallel import BatchShard
        sync = BatchShard(dist, rank, world)
    model = model.to(dev)
    opt = FusedAdam(model.parameters(), lr=1e-3, weight_decay=0)
    params = list(model.parameters())
    units = world if mode == 'dp' else 1             # batches of B the whole job consumes per synchronous step
    K, W = args.steps, args.warmup
    host_batches = [torch.from_numpy(b).pin_memory()
                    for b in make_batches(rows, cols, n_item, K + W, seed=2023 + (1000 * rank if mode == 'dp' else 0))]
    dev_batches = [b.to(dev) for b in host_batches]

    flag = torch.zeros(BATCH, dtype=torch.int64, device=dev)

    def as_batch(b):
        return [b[0], b[1], b[2], flag] if model_name == 'ncl' else [b[0], b[1], b[2]]
    if model_name == 'ncl':
        model.kmeans.iters = 20                      # the clustering runs once, before the timed region (ncl.py:73-74)
        model._cluster()

    last = {}

    def step_resident(i):
        opt.zero_grad()
        b = dev_batches[i % len(dev_batches)]
        loss, parts = model.cal_loss(as_batch(b))
        loss.backward()
        if sync is not None:
            sync.average_gradients(params)
        opt.step()
        last['loss'], last['parts'] = loss, parts
        return loss

    e2e_sampler = [None]
    from sslrec_b200.trainer import LossReader
    reader = LossReader(dev)
    seen = [0]

    def step_e2e_async(i):
        """The loop of sslrec_b200.trainer.Trainer.train_epoch: H2D of the batch, cal_loss, backward, step, and the
        step's loss scalars copied device -> pinned host asynchronously (read one step later)."""
        opt.zero_grad()
        b = host_batches[i % len(host_batches)].to(dev, non_blocking=True)
        loss, parts = model.cal_loss(as_batch(b))
        loss.backward()
        if sync is not None:
            sync.average_gradients(params)
        opt.step()
        if e2e_sampler[0] is not None:
            e2e_sampler[0].sample()
        seen[0] += len(reader.push(loss, parts))

    def step_e2e(i):
        opt.zero_grad()
        b = host_batches[i % len(host_batches)].to(dev, non_blocking=True)           # trainer.py:64
        loss, parts = model.cal_loss(as_batch(b))
        v = loss.item()                                          # trainer.py:66 (D2H sync)
        loss.backward()
        if sync is not None:
            sync.average_gradients(params)
        opt.step()
        if e2e_sampler[0] is not None:
            e2e_sampler[0].sample()                              # GPU is busy with the backward pass here
        for name in parts:                                       # trainer.py:72
            float(parts[name].detach())
        return v

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    timing_log = []

    def timed(fn, inline_sampling=False, no_sampling=False, steps=None, tail=None):
        K = steps or args.steps
        for i in range(W):
            fn(i)
        barrier()
        sampler = ClockSampler(local_rank) if (rank == 0 and not no_sampling) else None
        e2e_sampler[0] = sampler if inline_sampling else None
        l0 = _lib.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_host = time.perf_counter()
        e0.record()
        for i in range(K):
            fn(W + i)
        if tail is not None:
            tail()                                               # e.g. drain the pending device->host loss reads
        e1.record()
        t_host = time.perf_counter() - t_host
        if sampler is not None and not inline_sampling:
            sampler.drain(e1)                                    # the host is ahead of the GPU: sample while it works
        barrier()
        e2e_sampler[0] = None
        launches = _lib.launch_count() - l0
        clocks = sampler.result() if sampler is not None else None
        ms = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        timing_log.append({'loop': fn.__name__, 'gpu_ms_per_step': ms / K, 'host_enqueue_ms_per_step': 1e3 * t_host / K,
                           'sampling': 'inline' if inline_sampling else ('none' if no_sampling else 'drain')})
        return ms / K, launches, clocks

    # burn-in: allocator cache, module loading, NCCL channels and GPU clocks settle before anything is timed
    for i in range(30):
        step_resident(i % (K + W))
    barrier()
    # the value is timed WITHOUT NVML traffic (sampling while a sub-millisecond-per-step workload runs stalls the GPU:
    # lightgcn-gowalla read 6.6 ms/step sampled vs 0.7 ms unsampled); the clocks come from an immediate sampled replay
    # Five passes of exactly K steps each; the value is the MEDIAN pass and every pass is listed in timing_log.  The GPU
    # work is deterministic; what varies is the host: the boxes are shared and cgroup-limited (r01: a pass read
    # 8.7 ms/step where its neighbours read 2.9 ms with identical kernels, see profiles/r01d_*).
    passes = sorted((timed(step_resident, no_sampling=True) for _ in range(5)), key=lambda p: p[0])
    ms_res, launches, _ = passes[2]                      # the MEDIAN pass is the value; all five are in timing_log
    ms_res_best = passes[0][0]
    dump = outputs_of_step(model, last['loss'], last['parts']) if (args.dump_outputs and rank == 0) else None
    ms_res_sampled, _, clocks = timed(step_resident)
    if clocks is not None:
        clocks['sampled_replay_ms_per_step'] = ms_res_sampled
    # e2e is timed WITHOUT clock sampling (one NVML sample costs ~14 ms of host time, which the per-step
    # syncs of this loop would expose); its clocks come from a short sampled replay of the same loop
    ms_e2e_strict = float(np.median([timed(step_e2e, no_sampling=True)[0] for _ in range(3)]))

    def timed_async():
        ms, _, _ = timed(step_e2e_async, no_sampling=True, tail=lambda: seen.__setitem__(0, seen[0] + len(reader.flush())))
        return ms
    ms_e2e = float(np.median([timed_async() for _ in range(5)]))
    _, _, clocks_e2e = timed(step_e2e, inline_sampling=True)

    # ---- live kernel timings (CUDA events on the launching stream) over K more steps ----
    engine.TIMER = engine.KernelTimer()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        step_resident(W + i)
    e1.record()
    barrier()
    prof_ms = e0.elapsed_time(e1) / K
    summ = engine.TIMER.summary()
    engine_launches = engine.TIMER.launches()
    engine.TIMER = None
    if os.environ.get('BENCH_DIAG'):
        timed(step_resident, no_sampling=True)
        timed(step_e2e, no_sampling=True)

    def assemble():
        """Rank 0: everything of the bench line except the row-shard record."""
        # ---- one real epoch through Trainer.train_epoch (sample_negs + loader + loop), device loader vs host DataLoader ----
        epoch = None
        if world == 1 and model_name != 'ncl' and len(rows) // BATCH <= 1000:
            try:
                import types
                from sslrec_b200.data_handler import DeviceLoader, DeviceTrnData
                from sslrec_b200.trainer import Trainer
                epoch = {'batches': (len(rows) + BATCH - 1) // BATCH,
                         'how': 'wall clock of Trainer.train_epoch (negative sampling, shuffling, batching, H2D, steps, loss reads), after one warm-up epoch'}
                import torch.utils.data as tdata
                epoch['loaders'] = ('device_loader = train.device_loader: true (pairs, negative sampling, shuffle and batching on the device); host_dataloader = the data '
                                    'handler\'s default (HostBatchLoader: the reference\'s DataLoader(shuffle=True) batch for batch, gathered by array indexing); '
                                    'torch_dataloader = torch.utils.data.DataLoader itself over the same dataset (the reference\'s data path)')
                for key, loader in (('device_loader', DeviceLoader(DeviceTrnData(trn, dev, 2023), BATCH)), ('host_dataloader', dh.train_dataloader),
                                    ('torch_dataloader', tdata.DataLoader(dh.train_dataloader.dataset, batch_size=BATCH, shuffle=True, num_workers=0))):
                    tr = Trainer(types.SimpleNamespace(train_dataloader=loader))
                    tr.optimizer = opt
                    best = None
                    for rep in range(2 if key == 'torch_dataloader' else 3):
                        torch.cuda.synchronize()
                        t0 = time.perf_counter()
                        tr.train_epoch(model, rep)
                        torch.cuda.synchronize()
                        dt = time.perf_counter() - t0
                        best = dt if (best is None or rep == 1) else min(best, dt)      # rep 0 is the warm-up
                    epoch[key + '_steps_per_sec'] = len(loader) / best
                    epoch[key + '_epoch_s'] = best
            except Exception as e:      # noqa: BLE001 -- an extra record must never cost the bench line
                epoch = {'error': repr(e)[:400]}

        # ---- one all-rank evaluation pass through Trainer.evaluate (full_predict + _mask_predict from the device CSR, native top-40, metrics on the
        # host; trainer.py:139-150 + metrics.py:82-127) over every user, one synthetic held-out item each ----
        evalrec = None
        if world == 1 and args.workload == 'simgcl-amazon':
            try:
                import types
                import torch.utils.data as tdata
                from sslrec_b200.data_handler import AllRankTstData
                from sslrec_b200.trainer import Trainer
                rs = np.random.RandomState(7)
                val = sp.coo_matrix((np.ones(n_user, dtype=np.float32), (np.arange(n_user), rs.randint(0, n_item, n_user))), shape=(n_user, n_item))
                ld = tdata.DataLoader(AllRankTstData(val, trn, dense_mask=False), batch_size=cfg['test']['batch_size'], shuffle=False, num_workers=0)
                tr = Trainer(types.SimpleNamespace())
                secs = []
                for rep in range(2):                                     # rep 0 warms up (first propagation in eval mode, truth CSR)
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    res = tr.evaluate(model, loader=ld)
                    torch.cuda.synchronize()
                    secs.append(time.perf_counter() - t0)
                evalrec = {'users': n_user, 'batches': len(ld), 'eval_batch': cfg['test']['batch_size'], 'k': cfg['test']['k'], 'seconds': secs[-1],
                           'users_per_sec': n_user / secs[-1], 'recall': [float(v) for v in res['recall']],
                           'how': 'wall clock of Trainer.evaluate over all users: ssl_predict_mask (training positives masked from the device CSR) + ssl_topk '
                                  'per 1024-user batch, D2H of the top-40 indices, vectorised recall / ndcg on the host'}
                model.train()
            except Exception as e:      # noqa: BLE001 -- an extra record must never cost the bench line
                evalrec = {'error': repr(e)[:400]}

        # ---- the same step captured in ONE CUDA graph (sslrec_b200.graphed.GraphedStep; `train.cuda_graph: true` in the trainer), measured in
        # its own process: a capture that fails must not be able to touch this process's CUDA / RNG state ----
        graphed = None
        if world == 1 and not args.no_cuda_graph and model_name in ('lightgcn', 'simgcl', 'sgl', 'directau'):
            try:
                cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'graph', '--workload', args.workload, '--steps', str(K), '--warmup', str(W)]
                env = {k: v for k, v in os.environ.items() if k not in ('RANK', 'LOCAL_RANK', 'WORLD_SIZE')}
                env['CUDA_VISIBLE_DEVICES'] = os.environ.get('CUDA_VISIBLE_DEVICES', str(local_rank)).split(',')[local_rank] if os.environ.get('CUDA_VISIBLE_DEVICES') else str(local_rank)
                r = subprocess.run(cmd, capture_output=True, text=True, timeout=420, env=env)
                lines = [ln for ln in r.stdout.strip().splitlines() if ln.startswith('{')]
                graphed = json.loads(lines[-1]) if lines else {'error': (r.stderr or 'no output')[-400:]}
            except Exception as e:      # noqa: BLE001 -- an extra record must never cost the bench line
                graphed = {'error': repr(e)[:400]}

        # ---- the evaluation-side kernels (full_predict + _mask_predict through both of its kernels, top-k, one k-means iteration) at the
        # amazon shape, in their own process (tools/minor_kernels.py): an extra record, never allowed to cost the bench line ----
        eval_kernels = None
        if world == 1 and not args.no_eval_kernels and args.workload == 'simgcl-amazon':
            try:
                env = {k: v for k, v in os.environ.items() if k not in ('RANK', 'LOCAL_RANK', 'WORLD_SIZE')}
                r = subprocess.run([sys.executable, os.path.join(ROOT, 'tools', 'minor_kernels.py')], capture_output=True, text=True, timeout=240, env=env)
                lines = [ln for ln in r.stdout.strip().splitlines() if ln.startswith('{')]
                eval_kernels = json.loads(lines[-1]) if lines else {'error': (r.stderr or 'no output')[-400:]}
            except Exception as e:      # noqa: BLE001
                eval_kernels = {'error': repr(e)[:400]}

        peaks, peak_kind = measured_peaks()
        N, nnz, d = n_user + n_item, 2 * len(rows), hp['embedding_size']
        L = hp['layer_num']
        views = n_views(model_name)
        launches_all = engine_launches

        def prop_alg_bytes(m):
            """Algorithmic bytes of one propagation launch (DESIGN.md section 4): per stored entry its (col, val) pair
            (8 B) and one d-wide row per gathered view (4 d B); per output row its work item (16 B), every d-wide
            row the epilogue must read (residual, layer-sum sources, regulariser row) and every row it writes."""
            row = 4 * m['dim']
            b = m['nnz'] * (8 + row * m['gather_views'])
            per_row = 16 + (row * m['views'] if m['residual'] else 0) + sum(row * sv for sv in m['sum_src']) + (row if m['reg_src'] else 0)
            per_row += row * m['views'] if m['x_out'] else 0
            per_row += (row if m['reduce_views'] else row * m['views']) if m['sum_out'] else 0
            return b + m['rows'] * per_row
        def prop_min_bytes(m):
            """Compulsory HBM bytes of the same launch (SURVEY.md 8d bytes_min): every distinct input row ONCE per gathered
            view (n_cols rows, not nnz), the CSR once, and the same per-row epilogue reads / writes."""
            row = 4 * m['dim']
            per_row = 16 + (row * m['views'] if m['residual'] else 0) + sum(row * sv for sv in m['sum_src']) + (row if m['reg_src'] else 0)
            per_row += row if m.get('reg_src2') else 0
            per_row += row * m['views'] if m['x_out'] else 0
            per_row += (row if m['reduce_views'] else row * m['views']) if m['sum_out'] else 0
            return N * row * m['gather_views'] + 8 * m['nnz'] + m['rows'] * per_row
        prop = [(m, ms) for name, m, ms in launches_all if name in ('prop_fwd', 'prop_bwd')]
        prop_ms = sum(ms for _, ms in prop)
        prop_bytes = sum(prop_alg_bytes(m) for m, _ in prop)
        prop_min = sum(prop_min_bytes(m) for m, _ in prop)
        secs = prop_ms * 1e-3
        gather_rate = prop_bytes / secs / 1e9 if prop else None           # counts a gathered row once per stored entry: L2 hits included
        achieved = prop_min / secs / 1e9 if prop else None                # bytes that MUST cross HBM / time
        traffic = ncu_traffic('prop_kernel', f'views{views}_dim{d}_{graph}')
        gpeak = ncu_traffic('gather_peaks', 'l2_resident_GBps')           # measured by tools/gather_bench on this pool (profiles/)
        n_l = len(prop) if prop else 1
        roofline = {'kernel': 'prop_kernel (ssl_propagate_layer; all forward + transposed-backward launches of the timed steps)',
                    'bound': 'hbm', 'achieved': achieved, 'peak': peaks['hbm_gbs'], 'peak_kind': peak_kind + ' (burst copy)', 'unit': 'GB/s',
                    'frac': (achieved / peaks['hbm_gbs']) if achieved else None,
                    'frac_min': (achieved / peaks['hbm_gbs']) if achieved else None,
                    'frac_dram': (traffic / (secs / n_l) / 1e9 / peaks['hbm_gbs']) if (traffic and prop) else None,
                    'traffic': traffic, 'traffic_over_min': (traffic / (prop_min / n_l)) if (traffic and prop) else None,
                    'min_bytes_per_launch': prop_min / n_l if prop else None,
                    'l2_inclusive_gather_GBps': gather_rate, 'gather_bytes_per_launch': prop_bytes / n_l if prop else None,
                    'l2_gather_peak_GBps': gpeak, 'frac_l2_gather': (gather_rate / gpeak) if (gpeak and gather_rate) else None,
                    'avg_launch_ms': prop_ms / n_l if prop else None,
                    'launches_per_step': len(prop) / K, 'share_of_step': prop_ms / K / prof_ms if prof_ms else None,
                    'note': 'achieved / frac / frac_min = compulsory bytes (each input row once, CSR once, epilogue rows) over the live CUDA-event time: '
                            'the HBM roofline; frac_dram = ncu dram bytes of the committed capture over the same time; l2_inclusive_gather_GBps counts a '
                            'gathered row once per stored entry (what the SMs pull through the L2: bounded by the L2 gather rate, not by HBM)'}
        # the dense InfoNCE contraction (not HBM-bound): on the tcgen05 tensor cores with 3xTF32 error compensation when
        # dim is 32 / 64, else on the FP32 FMA pipe
        nce = [(m, ms) for name, m, ms in launches_all if name in ('nce_gemm_fwd', 'nce_gemm_bwd')]
        nce_ms = sum(ms for _, ms in nce)
        nce_flops_step = sum(4.0 * m['B'] * m['n'] * m['dim'] for m, _ in nce) / K          # fp32-equivalent: S = R C^T and O += E C
        sm_mhz = (clocks or {}).get('sm_mhz') or 1965.0
        roofline_nce = None
        if nce:
            used_tc = all(m.get('tc') for m, _ in nce)
            eq_tf = nce_flops_step * K / (nce_ms * 1e-3) / 1e12
            if used_tc:
                peak = peaks['bf16_tflops'] / 2.0
                roofline_nce = {'kernel': 'softmax_gemm_tc_kernel (ssl_softmax_gemm_tf32x3, forward + backward launches)', 'bound': 'tensor',
                                'achieved': 3.0 * eq_tf, 'peak': peak, 'unit': 'TFLOP/s', 'frac': 3.0 * eq_tf / peak,
                                'peak_kind': peak_kind + ' cuBLAS bf16 burst / 2 (kind::tf32 issues at half the bf16 rate)',
                                'fp32_equivalent_tflops': eq_tf, 'mma_flop_per_step': 3.0 * nce_flops_step,
                                'note': 'three tf32 products per fp32-grade product (3xTF32)', 'share_of_step': nce_ms / K / prof_ms,
                                'traffic': ncu_traffic('softmax_gemm_tc_kernel', f'dim{d}_{graph}')}
            else:
                fp32_peak = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12
                roofline_nce = {'kernel': 'softmax_gemm_kernel (ssl_softmax_gemm, forward + backward launches)', 'bound': 'fp32_fma', 'achieved': eq_tf,
                                'peak': fp32_peak, 'peak_kind': f'148 SM x 128 FMA/clk x 2 x {sm_mhz:.0f} MHz', 'unit': 'TFLOP/s',
                                'frac': eq_tf / fp32_peak, 'flop_per_step': nce_flops_step, 'share_of_step': nce_ms / K / prof_ms}
        n_prop_layers = max(L, 2 * hp.get('high_order', 0))
        emb_per_step = 2.0 * views * n_prop_layers * nnz if model_name != 'sgl' else 2.0 * L * nnz * (1 + 2 * hp['keep_rate'])

        # ---- CPU baseline on this box's host cores (bounded sample) ----
        cpu = None
        # rank 0, N = 1 only (the N > 1 lines of the scaling series carry null)
        if world == 1 and not args.no_cpu_baseline and not graph.startswith('synthetic-xl'):
            try:
                line = cpu_baseline_subprocess(args.workload, 2, 45.0)
                cpu = dict(line.get('cpu_baseline') or {'error': line.get('unavailable')})
                if line.get('cpu_baseline') and hp.get('keep_rate', 1.0) == 1.0:
                    # "tuned CPU": the same step with the adjacency in CSR, so the GPU ratio is not flattered by the COO layout
                    try:
                        t2 = cpu_baseline_subprocess(args.workload, 1, 30.0, csr=True)['cpu_baseline']
                        cpu['tuned_csr'] = {'value': t2['value'], 'unit': 'steps/s', 'cores': t2['cores'], 'sample': t2['sample']}
                    except Exception as e:      # noqa: BLE001 -- a baseline extra must never cost the bench line
                        cpu['tuned_csr'] = {'error': repr(e)[:300]}
            except Exception as e:      # noqa: BLE001
                cpu = {'error': repr(e)[:300]}

        value = units * 1e3 / ms_res
        out = {
            'metric': 'train_steps_per_sec', 'value': value, 'unit': 'steps/s', 'n_gpus': world, 'steps': K, 'warmup': W,
            'ms_per_step': ms_res, 'higher_is_better': True, 'scaling': scaling_label(args.parallel, args.workload, n_user, n_item, world), 'vs_baseline': None, 'dtype': 'f32',
            'data': 'synthetic', 'config': workload_config(args.workload, n_user, n_item, len(rows), world, mode),
            'batches_per_sync_step': units, 'optimizer_steps_per_sec': 1e3 / ms_res,
            'e2e': {'value': units * 1e3 / ms_e2e, 'unit': 'steps/s', 'ms_per_step': ms_e2e, 'h2d_bytes_per_step': 3 * BATCH * 8,
                    'd2h_bytes_per_step': 4 * (1 + {'simgcl': 3, 'sgl': 3, 'lightgcn': 2}.get(model_name, 3)),
                    'how': 'sslrec_b200.trainer.Trainer.train_epoch loop: pinned-host batch -> H2D, cal_loss, backward, FusedAdam.step, '
                           'loss + loss terms copied D2H asynchronously and read one step later (all reads drained inside the timed region)',
                'strict_sync_value': units * 1e3 / ms_e2e_strict, 'strict_sync_ms_per_step': ms_e2e_strict,
                'strict_sync_how': 'the reference trainer\'s own loop: blocking loss.item() after cal_loss and float(v) per loss term (trainer.py:66,72)'},
            'e2e_strict_sync': {'value': units * 1e3 / ms_e2e_strict, 'unit': 'steps/s', 'ms_per_step': ms_e2e_strict,
                                'how': 'the reference trainer\'s blocking reads: loss.item() after cal_loss and float(v) per loss term (trainer.py:66,72)'},
            'e2e_epoch': epoch, 'e2e_eval': evalrec,
            'gpu_launches': launches, 'gpu_launches_per_step': launches / K,
            'embeddings_propagated_per_sec': emb_per_step * value,
            'roofline': roofline, 'roofline_infonce': roofline_nce, 'cpu_baseline': cpu, 'row_shard': None, 'cuda_graph': graphed, 'eval_kernels': eval_kernels,
            'roofline_note': 'roofline = the SpMM BASELINE.json names (HBM-bound); roofline_infonce = the kernel with the largest share of this '
                             'step (tensor-bound contraction); both carry share_of_step',
            'clocks': clocks, 'clocks_e2e': clocks_e2e, 'kernel_ms_per_step': {k: v['ms'] / K for k, v in summ.items()}, 'profiled_ms_per_step': prof_ms,
            'timing_log': timing_log, 'host': {'cpu_count': os.cpu_count(), 'affinity': len(os.sched_getaffinity(0)), 'loadavg': os.getloadavg(),
                                                  'usable_cpus': usable_cpus()},
        }
        return out

    out = assemble() if rank == 0 else None
    torch.cuda.synchronize()
    if dump is not None:
        write_outputs(args.dump_outputs, dump)
        del dump

    # ---- north_star's partition next to the data-parallel headline: the row-sharded LightGCN step on the config-4 graph
    # family scaled to N/8 (bench_rowshard.py), on every --gpus N line of the default workload ----
    row_shard = None
    want_leg = args.row_shard == 'on' or (args.row_shard == 'auto' and args.workload == 'simgcl-amazon')
    if want_leg:
        del model, opt, params, dev_batches, host_batches
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        def fallback():
            if rank != 0:
                return None
            out['row_shard'] = {'error': f'abandoned after {args.row_shard_deadline:.0f} s (a rank wedged inside the leg)'}
            return json.dumps(out)
        dog = Watchdog(args.row_shard_deadline, fallback)
        try:
            import bench_rowshard
            row_shard = bench_rowshard.leg(dist, rank, world, dev, steps=K, warmup=W,
                                           log=(lambda m: print('[row_shard] ' + m, file=sys.stderr, flush=True)) if rank == 0 else (lambda m: None))
        except Exception as e:      # noqa: BLE001 -- the leg is an extra record; it must never cost the bench line
            row_shard = {'error': repr(e)[:500]}
            if world > 1:
                print(f'[row_shard] rank {rank}: {e!r}', file=sys.stderr, flush=True)
    else:
        dog = None

    if rank == 0:
        out['row_shard'] = row_shard
        print(json.dumps(out), flush=True)
    if dog is not None:
        dog.cancel()
    if dist is not None:
        dist.destroy_process_group()


def run_graph(args):
    """--impl graph: the workload's training step through sslrec_b200.graphed.GraphedStep (one CUDA graph launch per step); prints the
    `cuda_graph` record of the bench line.  Single GPU."""
    import importlib
    import scipy.sparse as sp
    import sslrec_b200  # noqa: F401
    from sslrec_b200.config import default_config, load_config
    from sslrec_b200.data_handler import DataHandlerGeneralCF
    from sslrec_b200.graphed import GraphedStep
    from sslrec_b200.optim import FusedAdam
    from sslrec_b200.trainer import LossReader
    torch.cuda.set_device(0)
    torch.set_num_threads(min(4, torch.get_num_threads()))
    dev = torch.device('cuda', 0)
    model_name, graph, hp = WORKLOADS[args.workload]
    rows, cols, n_user, n_item = graph_arrays(graph)
    cfg = default_config(model_name, **hp)
    cfg['train']['batch_size'] = BATCH
    load_config(base=cfg, device=str(dev))
    dh = DataHandlerGeneralCF(sp.coo_matrix((np.ones(len(rows), dtype=np.float32), (rows, cols)), shape=(n_user, n_item)))
    dh.load_data()
    mod = importlib.import_module('sslrec_b200.general_cf.' + model_name)
    cls = [getattr(mod, a) for a in dir(mod) if a.lower() == model_name][0]
    torch.manual_seed(2023)
    model = cls(dh).to(dev)
    opt = FusedAdam(model.parameters(), lr=1e-3, weight_decay=0)
    K, W = args.steps, max(args.warmup, 3)
    host_batches = [torch.from_numpy(b).pin_memory() for b in make_batches(rows, cols, n_item, K + W)]
    dev_batches = [b.to(dev) for b in host_batches]
    as_batch = lambda b: [b[0], b[1], b[2]]
    reader = LossReader(dev)
    gs = GraphedStep(model, opt, as_batch(dev_batches[0]), warmup=3)
    for i in range(10):
        gs(as_batch(dev_batches[i % len(dev_batches)]))
    res = {}
    for key, from_host in (('resident', False), ('e2e', True)):
        per = []
        for _ in range(5):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t_host = time.perf_counter()
            e0.record()
            for i in range(K):
                b = host_batches[(W + i) % len(host_batches)].to(dev, non_blocking=True) if from_host else dev_batches[(W + i) % len(dev_batches)]
                gl, gp = gs(as_batch(b))
                if from_host:
                    reader.push(gl, gp)
            if from_host:
                reader.flush()
            e1.record()
            t_host = time.perf_counter() - t_host
            torch.cuda.synchronize()
            per.append((e0.elapsed_time(e1) / K, 1e3 * t_host / K))
        per.sort()
        mid = per[len(per) // 2]
        res[key] = {'ms_per_step': mid[0], 'steps_per_sec': 1e3 / mid[0], 'host_ms_per_step': mid[1], 'passes_ms': [p[0] for p in per]}
    loss = float(gl.item())
    gs.close()
    print(json.dumps({'how': 'zero_grad + cal_loss + backward + FusedAdam.step captured once (3 eager warm-up steps), replayed per batch; the seeds of the in-kernel '
                             'augmentation and the Adam step count are device-resident, so training is identical to the eager loop '
                             '(tests/test_gpu_models.py::test_cuda_graph_step_equals_eager_step); median of 5 passes of K steps; e2e = batch from pinned host memory '
                             '+ asynchronous D2H of the loss scalars, all reads drained inside the timed region',
                      'workload': args.workload, 'steps': K, 'seeds_per_step': gs.n_seeds, 'last_loss': loss, **res}), flush=True)


def run_xl(args):
    """BASELINE.json configs[3]: LightGCN on the synthetic 10 M x 2 M / 300 M-edge graph, d = 128, row-sharded over the
    GPUs (strong scaling: the same graph at every N).  The bench line's value is the sharded step; rank 0's single-GPU run
    of the same graph is measured in the same process when N > 1 (``row_shard.baselines``)."""
    rank, local_rank, world = rank_world()
    import bench_rowshard as R
    import sslrec_b200  # noqa: F401
    from sslrec_b200 import _lib
    torch.cuda.set_device(local_rank)
    torch.set_num_threads(min(4, torch.get_num_threads()))
    dev = torch.device('cuda', local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=dev)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    l0 = _lib.launch_count()
    rec = R.leg(dist, rank, world, dev, steps=args.steps, warmup=max(args.warmup, 3), full=True, baselines=True,
                log=(lambda m: print('[xl] ' + m, file=sys.stderr, flush=True)) if rank == 0 else (lambda m: None))
    launches = _lib.launch_count() - l0
    if rank == 0:
        if sampler is not None:
            sampler.sample()
        peaks, peak_kind = measured_peaks()
        one = rec if world > 1 else rec['baselines']['one_gpu_config4']
        ms, spmm_ms, n_launch = one['ms_per_step'], one['spmm_ms'], max(1.0, one.get('spmm_launches', 2 * R.LAYERS))
        n_user, n_item, n_edge = R.EIGHTH[0] * 8, R.EIGHTH[1] * 8, R.EIGHTH[2] * 8
        nnz_rank = one.get('nnz_per_rank', one.get('nnz'))
        rows_rank = one.get('rows_per_rank', n_user + n_item)
        row = 4 * R.DIM
        t_launch = spmm_ms / n_launch * 1e-3
        gather = nnz_rank * (8 + row) + rows_rank * (16 + 2 * row)          # a gathered row once per stored entry + (col, val) + work item + one row read + one written
        minb = (n_user + n_item) * row + 8 * nnz_rank + rows_rank * (16 + 2 * row)      # every table row once (a rank's entries touch ~all of them), CSR once
        per_entry = ncu_traffic('prop_kernel', 'config4_dram_bytes_per_entry')         # ncu capture of the full-size launch (profiles/r02_ncu_kernels.md)
        traffic = per_entry * nnz_rank if per_entry else None
        achieved = (traffic if traffic else minb) / t_launch / 1e9
        gpeak = ncu_traffic('gather_peaks', 'hbm_random_GBps')
        out = {
            'metric': 'train_steps_per_sec', 'value': 1e3 / ms, 'unit': 'steps/s', 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
            'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': 'lightgcn training step on the synthetic config-4 graph (BASELINE.json configs[3])', 'model_name': 'lightgcn', 'graph': 'synthetic-xl',
                       'n_user': n_user, 'n_item': n_item, 'nnz': 2 * n_edge, 'batch': BATCH, 'global_batch': BATCH, 'dim': R.DIM, 'layers': R.LAYERS,
                       'parallelism': ('single GPU' if world == 1 else f'x{world}: rows of A and E sharded, all-gather of every layer output fused into the SpMM epilogue (NVLink peer stores)'),
                       'l2': 'no explicit flush: the 6.1 GB tables exceed the 126 MB L2 by 50x'},
            'e2e': {'value': 1e3 / one['e2e_ms_per_step'], 'unit': 'steps/s', 'ms_per_step': one['e2e_ms_per_step'], 'h2d_bytes_per_step': 3 * BATCH * 8, 'd2h_bytes_per_step': 4,
                    'how': 'batch from pinned host memory -> H2D, cal_loss, backward, (sharded) FusedAdam.step, loss.item() every step'},
            'gpu_launches': launches,
            'embeddings_propagated_per_sec': 2.0 * R.LAYERS * 2 * n_edge * 1e3 / ms,
            'roofline': {'kernel': 'prop_kernel (per rank, all forward + transposed-backward launches)', 'bound': 'hbm', 'achieved': achieved, 'peak': peaks['hbm_gbs'],
                         'peak_kind': peak_kind + ' (burst copy)', 'unit': 'GB/s', 'frac': achieved / peaks['hbm_gbs'], 'traffic': traffic,
                         'frac_dram': (traffic / t_launch / 1e9 / peaks['hbm_gbs']) if traffic else None, 'frac_min': minb / t_launch / 1e9 / peaks['hbm_gbs'],
                         'min_bytes_per_launch': minb, 'l2_inclusive_gather_GBps': gather / t_launch / 1e9, 'gather_bytes_per_launch': gather,
                         'hbm_random_gather_peak_GBps': gpeak, 'avg_launch_ms': spmm_ms / n_launch, 'share_of_step': spmm_ms / ms,
                         'note': 'achieved = DRAM bytes per launch (ncu capture of this launch shape, scaled by the stored entries) / live CUDA-event time; without a capture the '
                                 'compulsory bytes; l2_inclusive_gather_GBps counts a gathered row once per stored entry (the Zipf head of the item side is served from L2, so it '
                                 'exceeds the uniform-random HBM gather rate); row-sharded launches also carry the NVLink stores of the fused all-gather'},
            'cpu_baseline': None, 'row_shard': rec, 'clocks': sampler.result() if sampler is not None else None,
        }
        print(json.dumps(out), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference', 'graph'])
    ap.add_argument('--workload', default='simgcl-amazon', choices=sorted(WORKLOADS))
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-cuda-graph', action='store_true', help='skip the cuda_graph record (e.g. under a profiler)')
    ap.add_argument('--no-eval-kernels', action='store_true', help='skip the eval_kernels record (predict / top-k / k-means timings in a subprocess)')
    ap.add_argument('--cpu-budget', type=float, default=170.0, help='--impl reference: wall-clock budget of the timed CPU steps (s)')
    ap.add_argument('--cpu-csr', action='store_true', help='--impl reference: adjacency converted with to_sparse_csr() ("tuned CPU")')
    ap.add_argument('--row-shard', default='auto', choices=['auto', 'on', 'off'],
                    help="attach the row-sharded config-4-family record ('auto': on the default workload only)")
    ap.add_argument('--row-shard-deadline', type=float, default=420.0, help='seconds after which a wedged row-shard leg is abandoned')
    ap.add_argument('--parallel', default='auto', choices=['auto', 'dp', 'shard'],
                    help='N > 1: dp = one batch per GPU + gradient all-reduce (weak scaling); shard = one batch, table rows sharded')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last timed training step returned (loss, loss terms, updated parameters, a '
                         'seeded row sample of the gradients) as DIR/<name>.npy, float32, at most 64 MB; same arguments, same inputs')
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != 'ours' or args.workload == 'lightgcn-xl'):
        raise SystemExit('bench.py: --dump-outputs covers the training step of --impl ours (every workload but lightgcn-xl)')
    args.warmup = max(args.warmup, 3) if args.impl == 'ours' else args.warmup
    if args.impl == 'reference':
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit('bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)')
        if args.impl == 'graph':
            run_graph(args)
        elif args.workload == 'lightgcn-xl':
            run_xl(args)
        else:
            run_ours(args)


if __name__ == '__main__':
    main()
