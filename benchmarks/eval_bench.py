"""Eval-mode forward passes (batch-norm with the running statistics), the way ``Trainer.evaluate(running_stats=True)`` runs
them (``model.eval()``, ``torch.no_grad()``): the fused conv+BN units on lbt_bn_fwd_apply_running[_pooled] against the eager
eval path (``dfxp.FUSE_UNITS = False``: quantisers, then torch arithmetic for Normalization_q / Rescale_q / add / ReLU).

    python benchmarks/eval_bench.py [--reps 10] [--warmup 2] [--json FILE]

Per workload: ms per forward for each path (median over ``--reps`` alternating pairs, CUDA events around each forward and a
synchronise after it), images/s, algorithmic bytes per forward, and whether the two paths' logits are bit-equal at the timed
size.  The 224^2 workloads' activations are far larger than the 126 MB L2, so their forwards stream from HBM; ResNet-20's
per-layer tensors (16 MB of s8 mantissas, 65 MB fp32 at batch 1000) partly fit it.

Algorithmic bytes: every library launch counts the bytes it declares (``meta`` of lbt_b200._lib.call); every aten operator
that moves data reads each CUDA tensor argument once and writes its outputs once (views and allocations count nothing).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch
from torch.utils._python_dispatch import TorchDispatchMode
from torch.utils._pytree import tree_flatten

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from lbt_b200 import _lib, dfxp as D, models as M  # noqa: E402

# (name, constructor, kwargs, batch, image): ImageNet ResNets at 224^2 and ResNet-20 at evaluate()'s default batch
WORKLOADS = [
    ('resnet18_224_b256', M.Resnet18, dict(image=224, num_classes=1000), 256, 224),
    ('resnet20_32_b1000', M.CIFAR10_Resnet20, {}, 1000, 32),
    ('resnet50_224_b128', M.Resnet50, dict(image=224, num_classes=1000), 128, 224),
]

_NO_DATA = ('view', '_unsafe_view', 'permute', 'expand', 'empty', 'empty_like', 'empty_strided', 'as_strided', '_reshape_alias',
            'alias', 'detach', 'slice', 'select', 'unsqueeze', 'squeeze', 't', 'transpose', 'lift_fresh', 'set_',
            'resize_', 'is_same_size', '_local_scalar_dense')


class AtenBytes(TorchDispatchMode):
    """Sums the bytes of the CUDA tensors each data-moving aten operator reads and writes."""

    def __init__(self):
        super().__init__()
        self.bytes, self.ops = 0, {}

    def __torch_dispatch__(self, func, types, args=(), kwargs=None):
        out = func(*args, **(kwargs or {}))
        name = func.overloadpacket.__name__
        if name not in _NO_DATA:
            n = sum(t.numel() * t.element_size() for t in tree_flatten((args, kwargs, out))[0]
                    if isinstance(t, torch.Tensor) and t.is_cuda)
            self.bytes += n
            self.ops[name] = self.ops.get(name, 0) + 1
        return out


def algorithmic_bytes(model, X):
    """(bytes, {source: bytes}) of one eval forward on the current path."""
    prof = _lib.Profiler()
    _lib.profiler = prof
    try:
        with AtenBytes() as ab:
            model(X)
    finally:
        _lib.profiler = None
    lib = sum(v['bytes'] for v in prof.summary().values())
    return lib + ab.bytes, dict(library=lib, aten=ab.bytes, aten_ops=ab.ops)


def device_info():
    name = torch.cuda.get_device_name()
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', str(torch.cuda.current_device())],
                           capture_output=True, text=True, timeout=30)
        power = r.stdout.strip() or 'unknown'
    except Exception:
        power = 'unknown'
    return name, power


def seed_running_stats(model, rng):
    with torch.no_grad():
        for m in model.modules():
            if isinstance(m, D.Normalization_q):
                C = m.X_mean_running.numel()
                m.X_mean_running.copy_(torch.from_numpy((0.3 * rng.standard_normal(C)).astype(np.float32)))
                m.X_var_running.copy_(torch.from_numpy((0.3 + 1.5 * rng.random(C)).astype(np.float32)))


def run(name, ctor, kw, B, image, reps, warmup):
    torch.manual_seed(0)
    rng = np.random.default_rng(0)
    model = ctor(8, weight_decay=2e-4, seed=1, **kw).cuda()
    model.runtime.finalize('cuda')
    seed_running_stats(model, rng)
    model.eval()
    X = torch.from_numpy((rng.standard_normal((B, image, image, 3)) * 0.5).astype(np.float32)).cuda().permute(0, 3, 1, 2)
    paths = {'fused': True, 'eager': False}
    times = {p: [] for p in paths}
    logits, nbytes = {}, {}
    try:
        with torch.no_grad():
            for p, fused in paths.items():
                D.FUSE_UNITS = fused
                for _ in range(warmup):
                    model(X)
                nbytes[p] = algorithmic_bytes(model, X)
            torch.cuda.synchronize()
            for _ in range(reps):
                for p, fused in paths.items():
                    D.FUSE_UNITS = fused
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    out = model(X)
                    e1.record()
                    torch.cuda.synchronize()
                    times[p].append(e0.elapsed_time(e1))
                    logits[p] = out
    finally:
        D.FUSE_UNITS = True
    res = dict(workload=name, batch=B, image=image, reps=reps,
               bit_equal=bool(torch.equal(logits['fused'], logits['eager'])))
    for p in paths:
        ms = statistics.median(times[p])
        res[p] = dict(ms=round(ms, 3), ms_min=round(min(times[p]), 3), img_s=round(B / ms * 1e3, 1),
                      bytes=nbytes[p][0], bytes_library=nbytes[p][1]['library'], bytes_aten=nbytes[p][1]['aten'],
                      aten_ops=nbytes[p][1]['aten_ops'])
    res['speedup'] = round(res['eager']['ms'] / res['fused']['ms'], 3)
    del model, X, logits
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--only', default=None, help='comma-separated workload names')
    ap.add_argument('--json', default=None, help='also write the results to this file')
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('eval_bench needs a CUDA device')
    dev, power = device_info()
    print('device: %s, power limit: %s' % (dev, power))
    out = dict(device=dev, power_limit=power, results=[])
    for name, ctor, kw, B, image in WORKLOADS:
        if a.only and name not in a.only.split(','):
            continue
        r = run(name, ctor, kw, B, image, a.reps, a.warmup)
        out['results'].append(r)
        print('%-18s fused %8.3f ms %9.1f img/s %6.2f GB | eager %8.3f ms %9.1f img/s %6.2f GB | x%.2f | logits bit-equal: %s'
              % (name, r['fused']['ms'], r['fused']['img_s'], r['fused']['bytes'] / 1e9, r['eager']['ms'], r['eager']['img_s'],
                 r['eager']['bytes'] / 1e9, r['speedup'], r['bit_equal']), flush=True)
    print(json.dumps(out))
    if a.json:
        with open(a.json, 'w') as f:
            json.dump(out, f, indent=1)


if __name__ == '__main__':
    main()
