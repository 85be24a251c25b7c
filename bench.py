#!/usr/bin/env python
"""bench.py — quantised-training throughput of the DFXP hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port)

A "step" is one full training step (forward, loss, backward with quantised gradients, momentum SGD,
range controller) of the workload below on synthetic data.  N > 1 is launched by torchrun, one rank
per GPU, weak scaling (fixed per-GPU batch), gradient + overflow-counter all-reduce over NCCL.

Default workload (BASELINE.json configs[3], the one the metric's "@1/2/4/8" names and the largest that fits one GPU at its
stated batch): ResNet-18 composed from the reference's blocks, 224x224, batch 256 per GPU, 8-bit dynamic fixed point for
W/A/G, stochastic rounding everywhere (the reference's behaviour).  ``--workload resnet20 | cifar10 | resnet50 | resnet50_g8``
select configs[1] / configs[0] / configs[4] (8-bit W/A + 16-bit G) and its 8-bit-G variant.  The same JSON line carries the
two microbenchmark halves of the metric (configs[2]): ``quantize`` (lbt_quantize over 2^28 elements, GB/s and fraction of the
measured HBM peak) and ``gemm`` (lbt_gemm_i8 at 8192^3, TOPS, fraction of the int8 nominal and of torch._int_mm timed in the
same run).  Rank 0 prints ONE JSON line.

    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR

also writes what the last step of the first timed region computed as DIR/<name>.npy (see dump_outputs): the loss, and the
weights, momentum slots, gradients and ranges the step left behind.  Inputs, initial weights and noise are seeded, so two
builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

def measured_traffic(workload, entry):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of a kernel class, read at run time from the committed
    `ncu --set full` capture of this very command (profiles/traffic.json, written by benchmarks/ncu_traffic.py from the
    .ncu-rep): {"<workload>": {"<C-ABI entry>": {"bytes_per_launch": ..., "launches": ..., "source": "<csv>"}}}.
    None when no capture of that class is committed."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'traffic.json')) as f:
            row = json.load(f).get(workload, {}).get(entry)
        return (float(row['bytes_per_launch']), row.get('source')) if row else (None, None)
    except Exception:
        return None, None

WORKLOADS = {
    # name: (model ctor name, image, classes, default batch per GPU, bits, grad_bits)
    'resnet20': ('CIFAR10_Resnet20', 32, 10, 256, 8, None),
    'cifar10': ('CIFAR10_Model', 32, 10, 128, 8, None),
    'resnet18': ('Resnet18', 224, 1000, 256, 8, None),
    'resnet50': ('Resnet50', 224, 1000, 128, 8, 16),          # BASELINE config 5: 8-bit W/A + 16-bit G
    'resnet50_g8': ('Resnet50', 224, 1000, 128, 8, None),
}


_REAL_STDOUT = None


def guard_stdout():
    """Everything libraries print to fd 1 during the run (NCCL's version banner, for one) goes to stderr; the ONE JSON line is
    written to the real stdout by emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    data = (json.dumps(line) + '\n').encode()
    if _REAL_STDOUT is None:
        os.write(1, data)
    else:
        os.write(_REAL_STDOUT, data)


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError('must be at least 1, got %d' % v)
    return v


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=positive_int, default=20, help='timed steps of each timed region')
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='native', choices=['native', 'reference'])
    ap.add_argument('--workload', default='resnet18', choices=sorted(WORKLOADS))
    ap.add_argument('--batch', type=int, default=0, help='per-GPU batch (0 = the workload default)')
    ap.add_argument('--no-graph', action='store_true', help='do not capture the step in a CUDA graph')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-micro', action='store_true', help='skip the quantize / GEMM microbenchmark legs (configs[2])')
    ap.add_argument('--cpu-batch', type=int, default=0, help='batch of the CPU baseline sample (0 = same as GPU)')
    ap.add_argument('--no-pdl', action='store_true', help='A/B: launch without programmatic dependent launch edges')
    ap.add_argument('--no-overlap', action='store_true', help='A/B: weight-gradient kernels on the main stream (no side branch)')
    ap.add_argument('--breakdown', action='store_true', help='also print the per-kernel time table to stderr')
    ap.add_argument('--dump-launches', default='', help='write the per-launch device times of one step (CSV) to this file')
    ap.add_argument('--dump-outputs', default='', metavar='DIR',
                    help='write the outputs of the last timed step as DIR/<name>.npy (native path, rank 0)')
    a = ap.parse_args()
    if a.dump_outputs and a.impl != 'native':
        ap.error('--dump-outputs writes the outputs of the native path')
    return a


DUMP_CAP = 1 << 22      # elements per dumped array: 16 MiB each, so the three model-sized arrays + the small ones stay under 64 MiB


def dump_outputs(path, arrays):
    """Write every array of ``arrays`` (name -> numpy array) flattened as ``path/<name>.npy``: float32 stays float32,
    everything else (integer ranges, counters) becomes float64, which holds it exactly.  An array of more than DUMP_CAP
    elements is written as a fixed sample: the elements at DUMP_CAP sorted indices drawn by numpy's default_rng(0), the
    same indices for the same size, so two runs of the same workload compare element for element."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, v in arrays.items():
        v = np.ascontiguousarray(v).reshape(-1)
        if v.size > DUMP_CAP:
            v = v[np.sort(np.random.default_rng(0).choice(v.size, DUMP_CAP, replace=False))]
        np.save(os.path.join(path, name + '.npy'), v.astype(np.float32 if v.dtype == np.float32 else np.float64))


def describe(a, batch):
    name, image, classes, _, bits, gbits = WORKLOADS[a.workload]
    return {
        'workload': '%s %dx%dx3 batch %d/GPU, %d-bit dfxp W/A/G%s, stochastic rounding (Philox), SGD momentum 0.9 wd 2e-4'
                    % (name, image, image, batch, bits, '' if not gbits else ' (%d-bit G)' % gbits),
        'global_batch': batch * a.gpus,
        'parallelism': 'dp%d' % a.gpus,
        'l2': 'per-step working set (activations + gradients, >1 GB) exceeds the 126 MB L2; no explicit flush',
    }


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's path, all host threads
# ------------------------------------------------------------------------------------------------


def cpu_steps(a, batch, steps, warmup):
    import numpy as np
    import torch
    from oracle import dfxp as O
    name, image, classes, _, bits, gbits = WORKLOADS[a.workload]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    kw = dict(weight_decay=2e-4, noise=O.PhiloxNoise(0), seed=0, grad_bits=gbits)
    if name.startswith('Resnet'):
        kw.update(image=image, num_classes=classes)
    model = getattr(O, name)(bits, **kw)
    rng = np.random.default_rng(0)
    X = torch.from_numpy((rng.standard_normal((batch, image, image, 3)) * 0.5).astype(np.float32))
    y = torch.from_numpy(rng.integers(0, classes, batch))
    for _ in range(warmup):
        model.train_step(X, y)
    t0 = time.perf_counter()
    for _ in range(steps):
        model.train_step(X, y)
    dt = (time.perf_counter() - t0) / max(1, steps)
    return batch / dt, dt, cores


CPU_BATCH = {'resnet20': 0, 'cifar10': 0, 'resnet18': 8, 'resnet50': 4, 'resnet50_g8': 4}     # 0 = the GPU batch


def run_reference(a):
    """The reference's CPU path (the oracle port: TensorFlow 1.x cannot run here, SURVEY F10) on all host threads.  The
    reference is single-device (F11): with N > 1 the N shards of a global batch would be processed by the same host cores
    one after the other, so the whole-job imgs/s IS the single-run imgs/s; rank 0 alone measures it, on the native arm's
    config."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    batch = a.batch or WORKLOADS[a.workload][3]
    cpu_batch = a.cpu_batch or CPU_BATCH[a.workload] or batch
    ips, dt, cores = cpu_steps(a, cpu_batch, a.steps, a.warmup)
    cfg = describe(a, batch)
    sample = ('%d timed steps (after %d warm-up) of the oracle port (torch-CPU fp32 restatement of dynamic_fixed_point.py) on a '
              'bounded sample of the workload: batch %d per step, %.2f s/step; the host cores are shared by all %d shards, so '
              'imgs/s does not depend on N' % (a.steps, a.warmup, cpu_batch, dt, a.gpus))
    line = {
        'impl': 'reference', 'metric': 'quantized train imgs/sec', 'value': ips, 'unit': 'imgs/s', 'n_gpus': a.gpus,
        'steps': a.steps, 'warmup': a.warmup, 'ms_per_step': dt * 1e3, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32 (fake-quant on CPU)', 'data': 'synthetic', 'config': cfg,
        'cpu_baseline': {'value': ips, 'unit': 'imgs/s', 'cores': cores, 'kind': 'port', 'sample': sample},
        'e2e': {'value': ips, 'unit': 'imgs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
        'note': 'TensorFlow 1.x reference cannot run in this image (SURVEY.md F10); this is the CPU oracle port',
    }
    emit(line)


# ------------------------------------------------------------------------------------------------
# configs[2]: the two microbenchmark halves of the metric, timed in the same run
# ------------------------------------------------------------------------------------------------


def micro_legs(dev, hbm_peak):
    """quantize GB/s (2^28 fp32 elements -> s8 mantissas, Philox stochastic rounding, 5 B/element algorithmic) and int8 GEMM
    TOPS (8192^3, fp32 rescaling epilogue) with the stock cuBLASLt s8 GEMM (torch._int_mm) beside it.  CUDA events around
    back-to-back launches after warm-up; the 1 GiB quantiser input and the 3 x 64 MiB GEMM operands exceed / rotate past the
    126 MB L2."""
    import torch
    from lbt_b200 import gemm as G, quantizer as Q

    def timed(fn, reps):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e-3 / reps

    out = {}
    n = 1 << 28
    x = torch.randn(256, n // 256, device=dev)
    m = torch.empty(256, n // 256, dtype=torch.int8, device=dev)
    ib = torch.tensor(2, dtype=torch.int32, device=dev)
    cnt = Q.new_counters(dev)
    q = {}
    for key, mode in (('minmax_stats', Q.ROUND_PHILOX | Q.STATS_MINMAX), ('exact_counts', Q.ROUND_PHILOX)):
        t = timed(lambda: Q.quantize(x, 8, ib, mode=mode, seed=1, offset=Q.make_offset(3, 0), want_fp32=False,
                                     mant_kind=Q.MANT_S8, out_mant=m, counters=cnt, update_range=False), 10)
        q[key] = {'gbs': n * 5 / t / 1e9, 'us': t * 1e6, 'frac_hbm': n * 5 / t / 1e9 / hbm_peak}
    out['quantize'] = {
        'elements': n, 'bits': 8, 'rounding': 'stochastic (in-kernel Philox)', 'out': 's8 mantissas',
        'algorithmic_bytes_per_element': 5, 'gbs': q['minmax_stats']['gbs'], 'frac_hbm': q['minmax_stats']['frac_hbm'],
        'hbm_peak_gbs': hbm_peak, 'target_frac': 0.70,
        'statistics': 'min/max overflow statistics (LBT_STATS_MINMAX: what every layer call site uses, the reference\'s '
                      'target_overflow_rate is always 0); exact_counts = the C-ABI default the parity tests compare',
        'modes': q}
    del x, m
    torch.cuda.empty_cache()
    N = 8192
    ops = 2.0 * N ** 3
    pool = [(torch.randint(-128, 128, (N, N), dtype=torch.int8, device=dev),
             torch.randint(-128, 128, (N, N), dtype=torch.int8, device=dev)) for _ in range(2)]
    o32 = torch.empty(N, N, dtype=torch.float32, device=dev)
    it = [0]

    def ours():
        A, B = pool[it[0] & 1]
        it[0] += 1
        G.gemm_i8(A, B, exp_const=-14, out=o32)

    def stock():
        A, B = pool[it[0] & 1]
        it[0] += 1
        torch._int_mm(A, B.t())

    t_ours = timed(ours, 10)
    try:
        t_stock = timed(stock, 10)
    except Exception:
        t_stock = None
    out['gemm'] = {
        'shape': '8192^3 s8 x s8 -> s32 in TMEM, fp32 rescaling epilogue', 'tops': ops / t_ours / 1e12, 'us': t_ours * 1e6,
        'int8_nominal_tops': 4500.0, 'frac_nominal': ops / t_ours / 1e12 / 4500.0, 'target_frac': 0.60,
        'int_mm_tops': ops / t_stock / 1e12 if t_stock else None,
        'frac_of_int_mm': t_stock / t_ours if t_stock else None,
        'int_mm': 'torch._int_mm (cuBLASLt s8 x s8 -> s32, no epilogue) on the same operands in the same run'}
    del pool, o32
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------
# clocks sampler
# ------------------------------------------------------------------------------------------------


class Clocks:
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.lines:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
                power.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'power_w_max': max(power) if power else None, 'samples': len(sm), 'reasons': sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------


def run_native(a):
    import numpy as np
    import torch
    import torch.distributed as dist
    from lbt_b200 import _lib, models as M
    from lbt_b200.trainer import Trainer

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py --impl native needs a GPU: the DFXP path has no CPU fallback')
    torch.cuda.set_device(local)
    if world > 1:
        if os.environ.get('NCCL_DEBUG', '').upper() in ('', 'VERSION'):
            os.environ['NCCL_DEBUG'] = 'WARN'        # NCCL's "NCCL version ..." banner goes to stdout: keep it to ONE JSON line
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    assert world == a.gpus, 'launch with torchrun --nproc-per-node %d (WORLD_SIZE=%d)' % (a.gpus, world)
    dev = torch.device('cuda', local)

    name, image, classes, dbatch, bits, gbits = WORKLOADS[a.workload]
    batch = a.batch or dbatch
    kw = dict(weight_decay=2e-4, grad_bits=gbits, seed=0)
    if name.startswith('Resnet'):
        kw.update(image=image, num_classes=classes)
    torch.manual_seed(0)
    model = getattr(M, name)(bits, **kw).to(dev)
    trainer = Trainer(model, lr=1e-2, momentum=0.9)
    if a.no_pdl:
        _lib.lib().lbt_set_pdl(0)
    if a.no_overlap:
        model.runtime.overlap = False

    # synthetic data: a small pool of pinned host batches (NHWC fp32, like the reference's feed_dict)
    rng = np.random.default_rng(1234 + rank)
    pool = 4
    hostX = [torch.from_numpy((rng.standard_normal((batch, image, image, 3)) * 0.5).astype(np.float32)).pin_memory()
             for _ in range(pool)]
    hosty = [torch.from_numpy(rng.integers(0, classes, batch)).pin_memory() for _ in range(pool)]
    devX = [x.to(dev) for x in hostX]
    devy = [y.to(dev) for y in hosty]
    Xs = torch.empty(batch, image, image, 3, device=dev)          # static step input (NHWC memory)
    ys = torch.empty(batch, dtype=torch.int64, device=dev)
    Xs.copy_(devX[0])
    ys.copy_(devy[0])
    X_view = Xs.permute(0, 3, 1, 2)                               # logical NCHW, channels_last storage
    h2d = Xs.numel() * 4 + ys.numel() * 8

    def eager_step():
        return trainer.step(X_view, ys)

    # ---- warm-up (eager) + per-step launch count -------------------------------------------------
    for _ in range(2):
        loss = eager_step()
    torch.cuda.synchronize()
    l0 = _lib.launch_count()
    loss = eager_step()
    torch.cuda.synchronize()
    launches_per_step = _lib.launch_count() - l0

    # ---- eager step time (the same step, launched kernel by kernel through ctypes + autograd) ------
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        eager_step()
    e1.record()
    torch.cuda.synchronize()
    eager_ms = e0.elapsed_time(e1) / 3

    # ---- the product path: Trainer.capture() owns the CUDA graph of the whole step ----------------
    graph_ok = False
    if not a.no_graph:
        try:
            trainer.capture(X_view, ys, warmup=2)
            graph_ok = True
        except Exception as e:  # report, fall back to eager launches (still the CUDA path)
            if rank == 0:
                print('[bench] CUDA graph capture failed (%s: %s); timing eager launches' % (type(e).__name__, e), file=sys.stderr)
            torch.cuda.synchronize()

    def step():
        return trainer.step_graph() if graph_ok else eager_step()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    # ---- timed region 1: inputs resident in HBM ---------------------------------------------------
    for i in range(a.warmup):
        Xs.copy_(devX[i % pool]); ys.copy_(devy[i % pool])
        step()
    clocks = Clocks(local)
    barrier()
    if rank == 0:
        clocks.start()
        time.sleep(0.25)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    profile_region = os.environ.get('LBT_PROFILE_REGION') == '1'     # `ncu --profile-from-start off`: capture exactly these steps
    if profile_region:
        torch.cuda.profiler.start()
    e0.record()
    for i in range(a.steps):
        Xs.copy_(devX[i % pool]); ys.copy_(devy[i % pool])
        loss = step()
    e1.record()
    barrier()
    if profile_region:
        torch.cuda.profiler.stop()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    clk = clocks.stop() if rank == 0 else None
    ms_step = ms_total / a.steps
    value = batch * world / (ms_step * 1e-3)
    final_loss = float(loss)
    outputs = None
    if a.dump_outputs and rank == 0:     # copied now: the steps of the second timed region train on from here
        rt = model.runtime
        outputs = {'loss': loss.detach().float().reshape(1).cpu().numpy(), 'weights': trainer.flat_w.cpu().numpy(),
                   'momentum': trainer.flat_a.cpu().numpy(), 'gradients': trainer.flat_g.cpu().numpy(),
                   'ranges': rt.flat['ranges'].cpu().numpy(), 'step_counter': rt.dev_step.reshape(1).cpu().numpy()}

    # ---- timed region 2: end to end through the public API with HOST buffers ----------------------
    # every step: H2D copy of ITS inputs from pinned host memory (prefetched on a copy stream while the previous step runs,
    # lbt_b200.trainer.HostFeeder) and a D2H read of ITS loss (read by the host one step later) — all inside the timed region
    from lbt_b200.trainer import HostFeeder
    feeder = trainer.feeder() if graph_ok else HostFeeder(step, X_view, ys)
    hostX = [x.permute(0, 3, 1, 2) for x in hostX]          # logical NCHW views of the pinned NHWC batches (same memory)
    feeder.prefetch(hostX[0], hosty[0])
    for i in range(min(3, a.warmup)):
        feeder.prefetch(hostX[(i + 1) % pool], hosty[(i + 1) % pool])
        feeder.step()
    feeder.drain()
    # one batch is in flight from the warm-up; the timed loop copies exactly one batch per step
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    losses = []
    for i in range(a.steps):
        feeder.prefetch(hostX[(i + 1) % pool], hosty[(i + 1) % pool])      # H2D of a step's inputs from pinned memory
        losses.append(feeder.step())                                        # D2H of the previous step's loss
    losses.append(feeder.drain())                                           # ... and of the last one
    e1.record()
    barrier()
    wall = time.perf_counter() - t0
    lv = losses[-1]
    e2e_ms = max_over_ranks(max(e0.elapsed_time(e1), 0.0)) / a.steps
    e2e_value = batch * world / (e2e_ms * 1e-3)

    # ---- live per-kernel timing: the step is captured once more with an event pair around every C-ABI launch
    # (external event nodes), so each replay times every kernel back to back on the device, without host gaps ----
    nprof = 3
    prof = None
    try:
        prof = _lib.Profiler(external=True)
        s2 = torch.cuda.Stream()
        s2.wait_stream(torch.cuda.current_stream())
        pg = torch.cuda.CUDAGraph()
        _lib.profiler = prof
        with torch.cuda.graph(pg, stream=s2):
            eager_step()
            cal = [(prof.event(), prof.event()) for _ in range(4)]   # empty pairs: the cost of the event nodes themselves
            for ea, eb in cal:
                ea.record()
                eb.record()
        _lib.profiler = None
        torch.cuda.synchronize()
        acc = {}
        pg.replay()
        torch.cuda.synchronize()
        for _ in range(nprof):
            pg.replay()
            torch.cuda.synchronize()
            overhead = min(ea.elapsed_time(eb) for ea, eb in cal)
            for name, ea, eb, meta in prof.records:
                d = acc.setdefault(name, dict(launches=0, ms=0.0, bytes=0, ops=0))
                d['launches'] += 1
                d['ms'] += max(0.0, ea.elapsed_time(eb) - overhead)
                d['bytes'] += (meta or {}).get('bytes', 0)
                d['ops'] += (meta or {}).get('ops', 0)
        if a.dump_launches and rank == 0:
            with open(a.dump_launches, 'w') as f:
                f.write('# one %s step, per-launch device time from event nodes inside the replayed CUDA graph (event overhead %.2f us subtracted)\n'
                        % (a.workload, overhead * 1e3))
                f.write('index,entry,us,algorithmic_bytes,ops\n')
                for i, (name, ea, eb, meta) in enumerate(prof.records):
                    f.write('%d,%s,%.2f,%d,%d\n' % (i, name, max(0.0, ea.elapsed_time(eb) - overhead) * 1e3,
                                                   (meta or {}).get('bytes', 0), (meta or {}).get('ops', 0)))
        summ, timing_mode = acc, 'per-launch CUDA events inside a replayed graph of the step'
    except Exception as e:      # fall back to eager bracketing (includes host launch gaps on tiny kernels)
        _lib.profiler = None
        if rank == 0:
            print('[bench] graph-event profiling unavailable (%s: %s); eager events' % (type(e).__name__, e), file=sys.stderr)
        torch.cuda.synchronize()
        prof = _lib.Profiler()
        _lib.profiler = prof
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(nprof):
            eager_step()
        e1.record()
        _lib.profiler = None
        summ, timing_mode = prof.summary(), 'per-launch CUDA events, eager launches'
    peaks_path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(peaks_path):
        peak, peak_kind = json.load(open(peaks_path))['hbm_gbs'], 'measured (MEASURED_PEAKS.json hbm_gbs)'
    else:
        peak, peak_kind = 6650.0, 'fallback (B200_PROFILING.md)'
    ours_ms = sum(d['ms'] for d in summ.values()) / nprof
    breakdown = {}
    for k, d in sorted(summ.items()):
        row = {'launches': d['launches'] // nprof, 'ms_per_step': d['ms'] / nprof}
        if d['bytes'] and d['ms'] > 0:
            row['gbs'] = (d['bytes'] / 1e9) / (d['ms'] * 1e-3)
            row['frac_hbm'] = row['gbs'] / peak
        if d['ops'] and d['ms'] > 0:
            row['tops'] = (d['ops'] / 1e12) / (d['ms'] * 1e-3)
        breakdown[k] = row
    breakdown['other (torch pooling / loss / adds, gaps)'] = {'ms_per_step': max(0.0, ms_step - ours_ms)}
    # the dominant kernel class of the step (largest share of device time among the classes with a byte model)
    cands = [(d['ms'], k) for k, d in summ.items() if d['bytes'] and d['ms'] > 0]
    top = max(cands)[1] if cands else None
    q = summ.get(top, dict(launches=0, ms=0.0, bytes=0, ops=0))
    achieved = (q['bytes'] / 1e9) / (q['ms'] * 1e-3) if q['ms'] > 0 else 0.0
    gemm = summ.get('lbt_gemm_i8')
    gemm_tops = (gemm['ops'] / 1e12) / (gemm['ms'] * 1e-3) if gemm and gemm['ms'] > 0 else None
    conv_ops = sum(d['ops'] for k, d in summ.items() if d['ops'])
    conv_ms = sum(d['ms'] for k, d in summ.items() if d['ops'])
    conv_tops = (conv_ops / 1e12) / (conv_ms * 1e-3) if conv_ms > 0 else None     # every contraction of the step
    dp_mode = trainer.dp_mode

    # ---- after the timed regions: are the replicas still bit-identical? (weights, ranges, step counter) ----
    rt = model.runtime
    torch.cuda.synchronize()
    sums = torch.stack([trainer.flat_w.view(torch.int32).to(torch.int64).sum(),
                        rt.flat['ranges'].to(torch.int64).sum() * 1000003 + (rt.flat['ranges'].to(torch.int64) *
                                                                          torch.arange(1, len(rt.sites) + 1, device=dev)).sum(),
                        rt.dev_step.to(torch.int64).reshape(())])
    replicas_identical = None
    if world > 1:
        lo, hi = sums.clone(), sums.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        replicas_identical = bool(torch.equal(lo, hi))
    dp_error = trainer.dp.error() if trainer.dp is not None else None
    if world > 1:
        t = torch.tensor([dp_error or 0], dtype=torch.int64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dp_error = int(t)

    if rank != 0:
        _finish(world)
        return

    # ---- configs[2]: quantise GB/s and int8 GEMM TOPS, same run, N=1 only ----------------------------
    micro = None
    if world == 1 and not a.no_micro:
        torch.cuda.empty_cache()
        try:
            micro = micro_legs(dev, peak)
        except Exception as e:
            micro = {'error': '%s: %s' % (type(e).__name__, e)}

    # ---- CPU baseline (the oracle port on this box's host cores), N=1 only -------------------------
    cpu = None
    if world == 1 and not a.no_cpu_baseline:
        cpu_batch = a.cpu_batch or CPU_BATCH[a.workload] or batch
        ips, dt, cores = cpu_steps(a, cpu_batch, 2, 1)
        cpu = {'value': ips, 'unit': 'imgs/s', 'cores': cores, 'kind': 'port',
               'sample': '2 timed training steps (after 1 warm-up) of the oracle port at batch %d, %.2f s/step' % (cpu_batch, dt)}

    traffic, traffic_src = measured_traffic(a.workload, top)
    exchange = {
        'fused': 'lbt_dp_step: one kernel over NVLink peer memory (reduce-scatter by peer loads + SGD on the owned slice + '
                 'all-gather of the weights by peer stores + counter sum + range controller)',
        'nccl': 'NCCL all-reduce of gradients and counters + lbt_sgd_momentum + lbt_update_ranges',
        'unfused': 'single GPU: lbt_sgd_momentum + lbt_update_ranges'}[dp_mode] if world > 1 or dp_mode != 'fused' \
        else 'single GPU: lbt_dp_step (SGD + range controller + step counter in one launch)'
    line = {
        'metric': 'quantized train imgs/sec', 'value': value, 'unit': 'imgs/s', 'n_gpus': world, 'steps': a.steps,
        'warmup': a.warmup, 'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 's8/u8 mantissas, s32 accumulate (8-bit dfxp%s); fp32 master weights' % (', 16-bit gradients as s8/u8 halves' if gbits else ''),
        'data': 'synthetic',
        'config': describe(a, batch),
        'exchange': exchange,
        'dp_error': dp_error,
        'replicas_identical': replicas_identical,
        'clocks': clk,
        'e2e': {'value': e2e_value, 'unit': 'imgs/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 4,
                'ms_per_step': e2e_ms, 'wall_ms_per_step': wall / a.steps * 1e3,
                'how': 'Trainer.capture() + Trainer.feeder(): per-step H2D of the inputs prefetched on a copy stream, the step as '
                       'one graph launch, per-step D2H loss read one step later'},
        'gpu_launches': launches_per_step * a.steps,
        'launches_per_step': launches_per_step,
        'cuda_graph': graph_ok,
        'eager_ms_per_step': eager_ms,
        'roofline': {'bound': 'hbm', 'kernel': top, 'achieved': achieved,
                     'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak if peak else None,
                     'traffic': traffic, 'traffic_source': traffic_src,
                     'peak_kind': peak_kind, 'launches_per_step': q['launches'] // nprof,
                     'avg_launch_us': q['ms'] / max(1, q['launches']) * 1e3,
                     'share_of_step': (q['ms'] / nprof) / ms_step if ms_step else None,
                     'algorithmic_bytes_per_launch': q['bytes'] / max(1, q['launches']),
                     'timing': timing_mode,
                     'note': 'tensors of this workload are 1-17 MB: the kernels are launch/latency bound, far below the HBM roofline'
                             if a.workload in ('resnet20', 'cifar10') else None},
        'quantize': (micro or {}).get('quantize'),
        'gemm': (micro or {}).get('gemm'),
        'micro_error': (micro or {}).get('error'),
        'gemm_tops_in_step': gemm_tops,
        'conv_tops_in_step': conv_tops,
        'breakdown_ms': breakdown,
        'kernel_ms_per_step': ours_ms,
        'loss': final_loss,
        'cpu_baseline': cpu,
    }
    if a.breakdown:
        for k, d in breakdown.items():
            print('[breakdown] %-28s %s' % (k, d), file=sys.stderr)
    if outputs is not None:
        dump_outputs(a.dump_outputs, outputs)
    emit(line)
    _finish(world)


def _finish(world):
    """End of a rank.  With several ranks the NCCL communicator is referenced by the captured CUDA graph, and tearing
    the process group down under it has been seen to block forever (the measurement itself is complete): skip the
    teardown and leave with a hard exit once everything is flushed."""
    if world <= 1:
        return
    import torch
    torch.cuda.synchronize()
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)


if __name__ == '__main__':
    args = parse()
    guard_stdout()
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_native(args)
