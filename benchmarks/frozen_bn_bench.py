"""Training steps with frozen batch-norm statistics (``Model.freeze_bn_statistics``): a captured ``Trainer`` step in three
modes, in one process, alternating —

    train         normal training (batch statistics, two BN backward passes per layer)
    frozen_fused  frozen statistics on the fused units (eval-mode forward kernels with k2 saved, lbt_bn_bwd_running)
    frozen_eager  frozen statistics on the eager path (``dfxp.FUSE_UNITS = False``: quantisers, then torch arithmetic)

    python benchmarks/frozen_bn_bench.py [--reps 10] [--steps 5] [--json FILE]

Each mode has its own model and Trainer (same seed, one normal step first so the running statistics are non-trivial) and is
captured once (``Trainer.capture``, two warm-up steps); the three graphs are then replayed in turn: one timed sample =
``--steps`` replays between two CUDA events, followed by a synchronise; the table gives the median over ``--reps`` samples in
ms per step.
The 224^2 workloads' activations are far larger than the 126 MB L2, so their steps stream from HBM.

Algorithmic bytes per step: one eager step per mode, where every library launch counts the bytes it declares (``meta`` of
lbt_b200._lib.call) and every data-moving aten operator reads each CUDA tensor argument once and writes its outputs once.
BN backward kernel times: the same eager step with every library launch bracketed by CUDA events (lbt_b200._lib.Profiler),
summed per entry point.
"""
import argparse
import json
import os
import statistics
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from eval_bench import AtenBytes, device_info  # noqa: E402
from lbt_b200 import _lib, dfxp as D, models as M  # noqa: E402
from lbt_b200.trainer import Trainer  # noqa: E402

WORKLOADS = [
    ('resnet18_224_b256', M.Resnet18, dict(image=224, num_classes=1000), 256, 224, 1000),
    ('resnet20_32_b256', M.CIFAR10_Resnet20, {}, 256, 32, 10),
    ('resnet50_224_b128_g16', M.Resnet50, dict(image=224, num_classes=1000, grad_bits=16), 128, 224, 1000),
]
MODES = {'train': (False, True), 'frozen_fused': (True, True), 'frozen_eager': (True, False)}   # (frozen, FUSE_UNITS)
BN_BWD = ('lbt_bn_bwd_quant_stats', 'lbt_bn_bwd_apply', 'lbt_bn_bwd_running')


def set_mode(tr, mode):
    frozen, fused = MODES[mode]
    tr.freeze_bn_statistics(frozen)
    D.FUSE_UNITS = fused


def measure_step(tr, X, y):
    """(algorithmic bytes, {source: bytes}, {BN backward entry point: (launches, ms)}) of one eager step."""
    prof = _lib.Profiler()
    _lib.profiler = prof
    try:
        with AtenBytes() as ab:
            tr.step(X, y)
    finally:
        _lib.profiler = None
    summ = prof.summary()
    lib = sum(v['bytes'] for v in summ.values())
    bn = {k: (v['launches'], round(v['ms'], 3)) for k, v in summ.items() if k in BN_BWD}
    return lib + ab.bytes, dict(library=lib, aten=ab.bytes), bn


def run(name, ctor, kw, B, image, classes, reps, steps):
    rng = np.random.default_rng(0)
    X = torch.from_numpy((rng.standard_normal((B, image, image, 3)) * 0.5).astype(np.float32)).cuda()
    X = X.permute(0, 3, 1, 2).contiguous(memory_format=torch.channels_last)
    y = torch.from_numpy(rng.integers(0, classes, B)).cuda()
    trainers, captured, nbytes = {}, {}, {}
    try:
        for mode in MODES:
            torch.manual_seed(0)
            tr = Trainer(ctor(8, weight_decay=2e-4, seed=1, **kw).cuda(), lr=1e-2, momentum=0.9)
            D.FUSE_UNITS = True
            tr.step(X, y)                                # one normal step: the running statistics are non-trivial
            set_mode(tr, mode)
            nbytes[mode] = measure_step(tr, X, y)
            try:
                tr.capture(X, y, warmup=2)
                captured[mode] = True
            except Exception as e:        # a path that cannot be captured is timed as eager steps (reported as such)
                print('[frozen_bn_bench] %s %s: capture failed (%s: %s); timing eager steps' % (name, mode, type(e).__name__, e),
                      file=sys.stderr)
                captured[mode] = False
            trainers[mode] = tr
        times = {m: [] for m in MODES}
        torch.cuda.synchronize()
        for _ in range(reps):
            for mode, tr in trainers.items():
                set_mode(tr, mode)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(steps):
                    if captured[mode]:
                        tr.step_graph()
                    else:
                        tr.step(X, y)
                e1.record()
                torch.cuda.synchronize()
                times[mode].append(e0.elapsed_time(e1) / steps)
    finally:
        D.FUSE_UNITS = True
    res = dict(workload=name, batch=B, image=image, reps=reps, steps_per_sample=steps)
    for mode in MODES:
        ms = statistics.median(times[mode])
        res[mode] = dict(captured=captured[mode], ms=round(ms, 3), ms_min=round(min(times[mode]), 3), img_s=round(B / ms * 1e3, 1),
                         bytes=nbytes[mode][0], bytes_library=nbytes[mode][1]['library'], bytes_aten=nbytes[mode][1]['aten'],
                         bn_backward=nbytes[mode][2])
    res['frozen_fused_vs_train'] = round(res['frozen_fused']['ms'] / res['train']['ms'], 3)
    res['frozen_eager_vs_fused'] = round(res['frozen_eager']['ms'] / res['frozen_fused']['ms'], 3)
    del trainers, X
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--steps', type=int, default=5, help='graph replays per timed sample')
    ap.add_argument('--only', default=None, help='comma-separated workload names')
    ap.add_argument('--json', default=None, help='also write the results to this file')
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('frozen_bn_bench needs a CUDA device')
    dev, power = device_info()
    print('device: %s, power limit: %s' % (dev, power))
    out = dict(device=dev, power_limit=power, results=[])
    for name, ctor, kw, B, image, classes in WORKLOADS:
        if a.only and name not in a.only.split(','):
            continue
        r = run(name, ctor, kw, B, image, classes, a.reps, a.steps)
        out['results'].append(r)
        print('%-22s ' % name + ' | '.join('%s %8.3f ms %6.2f GB' % (m, r[m]['ms'], r[m]['bytes'] / 1e9) for m in MODES) +
              ' | frozen fused / train %.3f, eager / fused %.2f' % (r['frozen_fused_vs_train'], r['frozen_eager_vs_fused']),
              flush=True)
        for m in MODES:
            print('    %-13s BN backward launches (count, ms): %s' % (m, r[m]['bn_backward']), flush=True)
    print(json.dumps(out))
    if a.json:
        with open(a.json, 'w') as f:
            json.dump(out, f, indent=1)


if __name__ == '__main__':
    main()
