"""Eval mode (batch-norm with the running statistics, dfxp:616) on the fused kernels: lbt_bn_fwd_apply_running and
lbt_bn_fwd_apply_running_pooled against the eager eval path (``fused=False`` / ``FUSE_UNITS = False``) and the exact
oracle in inference mode.  The arithmetic is the training kernels' with another source of mean and variance, so every
result is compared with torch.equal."""
import contextlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import dfxp as O

pytestmark = pytest.mark.gpu

from lbt_b200 import _lib, dfxp as D, models as M  # noqa: E402
from lbt_b200.trainer import Trainer  # noqa: E402

SEED = 77
RUN, RUN_POOLED = 'lbt_bn_fwd_apply_running', 'lbt_bn_fwd_apply_running_pooled'


def nchw(x_nhwc):
    return x_nhwc.permute(0, 3, 1, 2).cuda()


def nhwc(x_nchw):
    return x_nchw.permute(0, 2, 3, 1).contiguous().cpu()


@contextlib.contextmanager
def launches():
    """Records (entry point, args) of every successful library call."""
    seen = []
    call, try_call = _lib.call, _lib.try_call

    def spy_call(fn, *a, **k):
        call(fn, *a, **k)
        seen.append((fn, a))

    def spy_try(fn, *a, **k):
        ok = try_call(fn, *a, **k)
        if ok:
            seen.append((fn, a))
        return ok

    _lib.call, _lib.try_call = spy_call, spy_try
    try:
        yield seen
    finally:
        _lib.call, _lib.try_call = call, try_call


def names(seen):
    return [fn for fn, _ in seen]


def oracle_set_training(om, flag):
    """Training or inference mode for every Normalization_q / Dropout_q of an oracle model, inside blocks too.  Returns the
    number of Normalization_q layers set, which the caller checks against the model (a container this walk does not know
    would otherwise leave its batch-norms in training mode unnoticed)."""
    seen = []

    def walk(layer):
        if isinstance(layer, (O.Normalization_q, O.Dropout_q)):
            layer.train = flag
            seen.append(layer)
        for sub in getattr(layer, 'layers', ()):
            walk(sub)
        if isinstance(layer, O.ResidualBlock_q):
            walk(layer.residual)
            walk(layer.shortcut)
    for layer in om.layers:
        walk(layer)
    return sum(1 for m in seen if isinstance(m, O.Normalization_q))


def seed_bn(modules, rng):
    """Non-trivial running statistics, gamma and beta in every BatchNorm2d_q."""
    with torch.no_grad():
        for m in modules:
            if isinstance(m, D.BatchNorm2d_q):
                C = m[0].X_mean_running.numel()
                m[0].X_mean_running.copy_(torch.from_numpy((0.3 * rng.standard_normal(C)).astype(np.float32)))
                m[0].X_var_running.copy_(torch.from_numpy((0.3 + 1.5 * rng.random(C)).astype(np.float32)))
                m[1].gamma.copy_(torch.from_numpy((1 + 0.3 * rng.standard_normal(C)).astype(np.float32)))
                m[1].beta.copy_(torch.from_numpy((0.2 * rng.standard_normal(C)).astype(np.float32)))


# ---- BatchNorm2d_q alone ---------------------------------------------------------------------------------------------


@pytest.mark.parametrize('add', [False, True])
@pytest.mark.parametrize('C,H,B,relu', [(16, 8, 8, False), (64, 4, 16, True), (128, 7, 6, True), (32, 5, 33, False)])
def test_batchnorm_q_eval_fused_equals_eager_and_exact_oracle(C, H, B, relu, add):
    """lbt_bn_fwd_quant_stats + lbt_bn_fwd_apply_running vs fused=False (quantise, then torch arithmetic) vs the oracle in
    inference mode: outputs equal; running statistics, ranges and the step counter untouched; the range controller then
    takes the same decisions on all three."""
    rng = np.random.default_rng(C * 3 + H + B + add)
    ctx = O.Context(O.PhiloxNoise(SEED), exact=True)
    ol = O.BatchNorm_q(ctx, 'bn', 8, C, False, weight_decay=2e-4)
    rm = torch.from_numpy((0.3 * rng.standard_normal(C)).astype(np.float32))
    rv = torch.from_numpy((0.3 + 1.5 * rng.random(C)).astype(np.float32))
    g0 = torch.from_numpy((1 + 0.3 * rng.standard_normal(C)).astype(np.float32))
    b0 = torch.from_numpy((0.2 * rng.standard_normal(C)).astype(np.float32))
    ol.layers[0].X_mean_running, ol.layers[0].X_var_running = rm.clone(), rv.clone()
    ol.layers[1].gamma.data.copy_(g0)
    ol.layers[1].beta.data.copy_(b0)
    x = torch.from_numpy((rng.standard_normal((B, H, H, C)) * 1.2 + 0.3).astype(np.float32))
    a = torch.from_numpy((rng.standard_normal((B, H, H, C)) * 0.5).astype(np.float32)) if add else None
    y_o = ol.forward(x)
    if add:
        y_o = y_o + a
    if relu:
        y_o = torch.relu(y_o)
    outs, ranges = [], []
    for fused in (True, False):
        rt = D.Runtime(SEED)
        pl = D.BatchNorm2d_q(8, C, weight_decay=2e-4, runtime=rt, fused=fused).cuda()
        rt.finalize('cuda')
        with torch.no_grad():
            for t, v in ((pl[0].X_mean_running, rm), (pl[0].X_var_running, rv), (pl[1].gamma, g0), (pl[1].beta, b0)):
                t.copy_(v)
        pl.eval()
        r0, s0 = rt.flat['ranges'].clone(), rt.dev_step.clone()
        with torch.no_grad(), launches() as seen:
            y = pl(nchw(x), add=nchw(a) if add else None, relu=relu)
        assert (RUN in names(seen)) == fused
        outs.append(nhwc(y))
        assert torch.equal(pl[0].X_mean_running.cpu(), rm) and torch.equal(pl[0].X_var_running.cpu(), rv)
        assert torch.equal(rt.flat['ranges'], r0) and torch.equal(rt.dev_step, s0)
        rt.update_ranges()
        ranges.append(list(rt.ranges().values()))
    assert torch.equal(outs[0], outs[1]), int((outs[0] != outs[1]).sum())
    assert torch.equal(outs[0], y_o), int((outs[0] != y_o).sum())
    assert ranges[0] == ranges[1] == [int(q.range) for q in ol.quantizers()]


def test_batchnorm_q_eval_with_gradients_stays_eager():
    """Eval mode while autograd records a graph: no running-statistics kernel, and the backward pass works."""
    rt = D.Runtime(SEED)
    pl = D.BatchNorm2d_q(8, 16, runtime=rt).cuda()
    rt.finalize('cuda')
    seed_bn([pl], np.random.default_rng(0))
    pl.eval()
    x = torch.randn(4, 16, 6, 6, device='cuda').contiguous(memory_format=torch.channels_last).requires_grad_(True)
    with launches() as seen:
        y = pl(x)
        y.sum().backward()
    assert RUN not in names(seen) and 'lbt_bn_fwd_apply' not in names(seen)
    assert x.grad is not None and bool(torch.isfinite(x.grad).all())


# ---- fused units -----------------------------------------------------------------------------------------------------


def eval_both(rt, fn):
    """fn() in eval mode without gradients, on the fused path and with FUSE_UNITS off, from the same ranges, counters and
    step: [(output, ranges after the controller, launches)] for the two."""
    r0, c0, s0 = rt.flat['ranges'].clone(), rt.flat['counters'].clone(), rt.dev_step.clone()
    res = []
    for fused in (True, False):
        rt.flat['ranges'].copy_(r0)
        rt.flat['counters'].copy_(c0)
        rt.dev_step.copy_(s0)
        D.FUSE_UNITS = fused
        try:
            with torch.no_grad(), launches() as seen:
                out = fn()
        finally:
            D.FUSE_UNITS = True
        out = out.detach().clone()
        rt.update_ranges()
        res.append((out, rt.flat['ranges'].clone(), seen))
    (ya, ra, sa), (yb, rb, sb) = res
    assert torch.equal(ya, yb), int((ya != yb).sum())
    assert torch.equal(ra, rb)
    assert RUN not in names(sb) and RUN_POOLED not in names(sb) and 'lbt_bn_fwd_quant_stats' not in names(sb)
    return sa


def modules_on(rt, mods, rng):
    ml = torch.nn.ModuleList(mods).cuda()
    rt.finalize('cuda')
    seed_bn(ml.modules(), rng)
    ml.eval()
    return ml


def image(rng, shape, signed=True):
    x = torch.from_numpy((rng.standard_normal(shape) * 0.8).astype(np.float32))
    return (x if signed else x.abs()).cuda().contiguous(memory_format=torch.channels_last)


def test_unit_eval_hands_mantissas_to_the_next_conv():
    rng = np.random.default_rng(1)
    rt = D.Runtime(SEED)
    conv1 = D.Conv2d_q(8, 16, 32, 3, 1, 'SAME', bias=False, input_signed=False, runtime=rt, name='c1')
    bn1 = D.BatchNorm2d_q(8, 32, relu=True, runtime=rt, name='bn1')
    conv2 = D.Conv2d_q(8, 32, 32, 3, 1, 'SAME', bias=False, input_signed=False, runtime=rt, name='c2')
    modules_on(rt, [conv1, bn1, conv2], rng)
    x = image(rng, (4, 16, 8, 8), signed=False)
    hollow = []

    def fn():
        h = D.conv_bn_unit(conv1, bn1, x, next_conv=conv2, want_fp32=False)
        hollow.append(bool(getattr(h, '_lbt_hollow', False)))
        return conv2(h)

    seen = eval_both(rt, fn)
    assert hollow == [True, False]           # fused: the activation between the units exists only as mantissas
    runs = [a for fn_, a in seen if fn_ == RUN]
    assert len(runs) == 1 and runs[0][20] is None and runs[0][21] is None and runs[0][23] is not None   # no k2, no fp32 out


def test_strided_block_eval_feeds_both_consumers():
    """conv+BN+ReLU producing the input of a strided basic block: the producing kernel quantises it for the block's first 3x3
    and for its 1x1 shortcut convolution (the second consumer)."""
    rng = np.random.default_rng(2)
    rt = D.Runtime(SEED)
    conv0 = D.Conv2d_q(8, 16, 16, 3, 1, 'SAME', bias=False, input_signed=True, runtime=rt, name='c0')
    bn0 = D.BatchNorm2d_q(8, 16, relu=True, runtime=rt, name='bn0')
    blk = D.ResidualBlock_q(8, 16, 32, 2, runtime=rt, name='blk')
    modules_on(rt, [conv0, bn0, blk], rng)
    x = image(rng, (4, 16, 16, 16))
    seen = eval_both(rt, lambda: D.run_layers([conv0, bn0, blk], x))
    runs = [a for fn_, a in seen if fn_ == RUN]
    assert len(runs) == 4                                        # bn0, bn1, shortcut bn, bn2 (+ add + ReLU)
    assert sum(1 for a in runs if a[26] is not None) == 1        # q_next2
    assert sum(1 for a in runs if a[18] is not None) == 1        # the residual sum


def test_bottleneck_block_eval():
    rng = np.random.default_rng(3)
    rt = D.Runtime(SEED)
    conv0 = D.Conv2d_q(8, 16, 32, 3, 1, 'SAME', bias=False, input_signed=True, runtime=rt, name='c0')
    bn0 = D.BatchNorm2d_q(8, 32, relu=True, runtime=rt, name='bn0')
    blk = D.ResidualBottleneck_q(8, 32, 16, 2, runtime=rt, name='bott')
    modules_on(rt, [conv0, bn0, blk], rng)
    x = image(rng, (3, 16, 12, 12))
    seen = eval_both(rt, lambda: D.run_layers([conv0, bn0, blk], x))
    assert names(seen).count(RUN) == 5


@pytest.mark.parametrize('N,H', [(2, 32), (3, 36)])          # 36: 18 x 18 -> 9 x 9, ragged windows and tiles
def test_imagenet_stem_eval_pooled_kernel(N, H):
    """7x7/2 conv -> BN -> ReLU -> 3x3/2 max-pool (C = 64) -> the next conv: one running-statistics kernel applies BN, ReLU,
    the pool and the consumer's input quantiser."""
    rng = np.random.default_rng(4)
    rt = D.Runtime(SEED)
    conv = D.Conv2d_q(8, 3, 64, 7, 2, 'SAME', bias=False, input_signed=True, runtime=rt, name='conv1')
    bn = D.BatchNorm2d_q(8, 64, relu=True, runtime=rt, name='conv1-bn')
    pool = D.MaxPool_q(3, 2, 'SAME')
    conv2 = D.Conv2d_q(8, 64, 64, 3, 1, 'SAME', bias=False, input_signed=False, runtime=rt, name='c2')
    modules_on(rt, [conv, bn, conv2], rng)
    x = image(rng, (N, 3, H, H))
    seen = eval_both(rt, lambda: D.run_layers([conv, bn, pool, conv2], x))
    assert names(seen).count(RUN_POOLED) == 1 and RUN not in names(seen) and 'lbt_maxpool_fwd' not in names(seen)


# ---- whole models ----------------------------------------------------------------------------------------------------


def build(name, image_size, classes):
    extra = dict(image=image_size, num_classes=classes) if name.startswith('Resnet') else {}
    om = getattr(O, name)(8, weight_decay=2e-4, noise=O.PhiloxNoise(5), seed=1, exact=True, **extra)
    pm = getattr(M, name)(8, weight_decay=2e-4, seed=5, **extra).cuda()
    for a, b in zip(om.variables(), pm.parameters()):
        b.data.copy_(a.detach())
    return om, pm


def batch(rng, n, image_size, classes):
    X = torch.from_numpy((rng.standard_normal((n, image_size, image_size, 3)) * 0.5).astype(np.float32))
    y = torch.from_numpy(rng.integers(0, classes, n))
    return X, y


@pytest.mark.parametrize('name,B,image_size,classes', [('CIFAR10_Resnet20', 8, 32, 10), ('Resnet18', 4, 64, 100),
                                                      ('Resnet50', 4, 64, 100)])
def test_eval_forward_after_training_bit_exact_vs_exact_oracle(name, B, image_size, classes):
    """Two training steps (running statistics move), then an eval forward at an evaluation step word: the logits equal the
    oracle's in inference mode bit for bit; the loss agrees to 1e-6 (its mean is summed in another order)."""
    rng = np.random.default_rng(13)
    om, pm = build(name, image_size, classes)
    tr = Trainer(pm, lr=1e-2, momentum=0.9)
    for _ in range(2):
        X, y = batch(rng, B, image_size, classes)
        om.train_step(X, y, lr=1e-2, momentum=0.9)
        tr.step(X.permute(0, 3, 1, 2).cuda(), y.cuda())
    X, y = batch(rng, B, image_size, classes)
    word = 0x80000000 | (2 << 12)
    assert oracle_set_training(om, False) == sum(1 for m in pm.modules() if isinstance(m, D.Normalization_q))
    om.ctx.noise.step = word
    want = om.forward(X)
    pm.eval()
    pm.runtime.dev_step.fill_(word)
    with torch.no_grad(), launches() as seen:
        got = pm(X.permute(0, 3, 1, 2).cuda())
    assert RUN in names(seen)
    got = got.cpu()
    assert torch.equal(got, want), int((got != want).sum())
    lo = float(F.cross_entropy(want, y))
    lp = float(pm.loss(got.cuda(), y.cuda()))
    assert abs(lo - lp) <= 1e-6 * max(1.0, abs(lo))


# ---- Trainer.evaluate and launches -----------------------------------------------------------------------------------


def _trained_resnet20(steps=2, batch_size=16):
    torch.manual_seed(3)
    pm = M.CIFAR10_Resnet20(8, weight_decay=2e-4, seed=9).cuda()
    tr = Trainer(pm, lr=1e-2, momentum=0.9)
    rng = np.random.default_rng(1)
    for _ in range(steps):
        X, y = batch(rng, batch_size, 32, 10)
        tr.step(X.permute(0, 3, 1, 2).cuda(), y.cuda())
    return pm, tr, rng


def test_trainer_evaluate_running_stats_changes_nothing_and_equals_eager():
    pm, tr, rng = _trained_resnet20()
    X, y = batch(rng, 40, 32, 10)
    X, y = X.permute(0, 3, 1, 2).cuda(), y.cuda()
    rt = pm.runtime

    def state():
        torch.cuda.synchronize()
        return ([tr.flat_w.clone(), tr.flat_a.clone(), rt.flat['ranges'].clone(), rt.flat['counters'].clone(), rt.dev_step.clone()] +
                [b.clone() for _, b in pm.named_buffers()])

    before = state()
    with launches() as seen:
        r1 = tr.evaluate(X, y, batch_size=16, running_stats=True)            # 16 + 16 + 8
    assert names(seen).count(RUN) > 0
    assert all(m.training for m in pm.modules())
    for a, b in zip(before, state()):
        assert torch.equal(a, b)
    assert tr.evaluate(X, y, batch_size=16, running_stats=True) == r1
    D.FUSE_UNITS = False
    try:
        with launches() as seen:
            r_eager = tr.evaluate(X, y, batch_size=16, running_stats=True)
    finally:
        D.FUSE_UNITS = True
    assert RUN not in names(seen)
    assert r_eager == r1, (r_eager, r1)
    for a, b in zip(before, state()):
        assert torch.equal(a, b)


ARITH_OPS = {'aten::add', 'aten::add_', 'aten::sub', 'aten::sub_', 'aten::rsub', 'aten::mul', 'aten::mul_', 'aten::div',
             'aten::div_', 'aten::pow', 'aten::sqrt', 'aten::mean'}
ARITH_KERNELS = ('functor_add', 'mulfunctor', 'divfunctor', 'div_true', 'pow_', 'sqrt', 'meanops')


def test_eval_forward_launches_no_aten_arithmetic():
    """A ResNet-20 eval forward on the fused path calls no aten arithmetic and launches no aten arithmetic kernel (fills and
    copies are allowed); the eager eval path does both, which is what this check would see."""
    pm, _, rng = _trained_resnet20(steps=1)
    pm.eval()
    X = batch(rng, 32, 32, 10)[0].permute(0, 3, 1, 2).cuda()

    def profile(fused):
        D.FUSE_UNITS = fused
        try:
            with torch.no_grad():
                pm(X)
                torch.cuda.synchronize()
                with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU,
                                                        torch.profiler.ProfilerActivity.CUDA]) as prof:
                    pm(X)
                    torch.cuda.synchronize()
        finally:
            D.FUSE_UNITS = True
        events = prof.events()
        ops = {e.name for e in events} & ARITH_OPS
        kernels = {e.name for e in events if e.device_type == torch.autograd.DeviceType.CUDA and 'at::native' in e.name and
                   any(k in e.name.lower() for k in ARITH_KERNELS)}
        lbt = {e.name for e in events if e.device_type == torch.autograd.DeviceType.CUDA and 'bn_fwd2_kernel' in e.name}
        return ops, kernels, lbt

    ops, kernels, lbt = profile(True)
    assert not ops, ops
    assert not kernels, kernels
    assert lbt
    ops, kernels, _ = profile(False)
    assert ops and kernels
