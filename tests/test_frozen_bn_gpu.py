"""Training with frozen batch-norm statistics (BatchNorm2d_q.freeze_statistics / Model.freeze_bn_statistics) on the fused
kernels: the eval-mode forward kernels with k2 saved, and ONE backward launch per layer (lbt_bn_bwd_running), against the
eager path (``fused=False`` / ``FUSE_UNITS = False``) and the exact oracle with its batch-norms built with training=False.
Everything but the eager path's fp32 reductions is compared with torch.equal."""
import contextlib

import numpy as np
import pytest
import torch

from oracle import dfxp as O

pytestmark = pytest.mark.gpu

from lbt_b200 import _lib, data as PD, dfxp as D, models as M  # noqa: E402
from lbt_b200.trainer import Trainer  # noqa: E402

SEED = 77
WD = 2e-4
BWD = 'lbt_bn_bwd_running'
TRAINING_BN = ('lbt_bn_bwd_apply', 'lbt_bn_bwd_quant_stats', 'lbt_bn_fwd_apply', 'lbt_bn_fwd_apply2', 'lbt_bn_fwd_apply_pooled')


def nchw(x_nhwc):
    return x_nhwc.permute(0, 3, 1, 2).cuda()


def nhwc(x_nchw):
    return x_nchw.detach().permute(0, 2, 3, 1).contiguous().cpu()


@contextlib.contextmanager
def launches():
    """Records the entry point of every successful library call."""
    seen = []
    call, try_call = _lib.call, _lib.try_call

    def spy_call(fn, *a, **k):
        call(fn, *a, **k)
        seen.append(fn)

    def spy_try(fn, *a, **k):
        ok = try_call(fn, *a, **k)
        if ok:
            seen.append(fn)
        return ok

    _lib.call, _lib.try_call = spy_call, spy_try
    try:
        yield seen
    finally:
        _lib.call, _lib.try_call = call, try_call


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


def oracle_norms(om):
    """Every Normalization_q of an oracle model in forward order, found through every Layer_q-valued attribute (and list of
    them) of every layer, whatever the container: the model's layer list, Sequential_q, the blocks' residual / shortcut."""
    seen, found = set(), []

    def walk(obj):
        if id(obj) in seen:
            return
        seen.add(id(obj))
        if isinstance(obj, O.Normalization_q):
            found.append(obj)
            return
        for v in vars(obj).values():
            for sub in (v if isinstance(v, (list, tuple)) else (v,)):
                if isinstance(sub, O.Layer_q):
                    walk(sub)
    for layer in om.layers:
        walk(layer)
    return found


def oracle_bn_training(om, flag):
    """Set the ``training`` flag every oracle Normalization_q was built with while the rest of the oracle model keeps
    training (frozen statistics from this step on); returns the layers, which the caller checks against the model."""
    norms = oracle_norms(om)
    for m in norms:
        m.train = flag
    return norms


# The oracle's den, (var + eps) ** 0.5, is torch's CPU square root, which is not correctly rounded for about 0.5 % of fp32
# inputs (torch 2.11, every CPU capability).  dfxp:616 on the device — torch's CUDA sqrt and the library alike — is
# RN(sqrt(RN(var + eps))).  In training mode the oracle's den only enters through quantised or batch-reduced values; with
# frozen statistics the VJP is g / den elementwise, so every element of an affected channel shows the oracle's error.
def cpu_den(var, eps=1e-5):
    return (var + eps) ** 0.5                                                           # the oracle's expression


def exact_den(var, eps=1e-5):
    v = var + eps                                                                       # fp32 add: correctly rounded
    return torch.from_numpy(np.sqrt(v.double().numpy()).astype(np.float32))             # fp64 sqrt rounded once: RN(sqrt)


def snap_running_var(var, eps=1e-5):
    """``var`` ([C], as the oracle holds it) moved up by a few ulps in every channel where torch's CPU sqrt misrounds
    ``var + eps``, so that the oracle's den is the correctly rounded one there too.  Returns (new var, channels moved)."""
    v = var.clone()
    bad = (cpu_den(v, eps) != exact_den(v, eps)).nonzero().flatten().tolist()
    for c in bad:
        for _ in range(256):
            v[c] = float(np.nextafter(np.float32(v[c]), np.float32(np.inf)))
            if bool(cpu_den(v, eps)[c] == exact_den(v, eps)[c]):
                break
    assert torch.equal(cpu_den(v, eps), exact_den(v, eps))
    return v, len(bad)


def running_buffers(modules):
    return [b.detach().clone() for m in modules for n, b in m.named_buffers() if 'running' in n]


# ---- BatchNorm2d_q alone ---------------------------------------------------------------------------------------------


@pytest.mark.parametrize('gbits', [8, 16])
@pytest.mark.parametrize('relu,add', [(False, False), (True, False), (True, True)])
@pytest.mark.parametrize('C', [16, 64, 256])
def test_batchnorm_q_frozen_fused_equals_eager_and_exact_oracle(C, relu, add, gbits):
    """Forward + backward of a frozen BatchNorm2d_q: fused (lbt_bn_fwd_apply_running with k2 + lbt_bn_bwd_running) against
    fused=False (Normalization_q honouring ``frozen``) and the exact oracle with training=False.  Output, dx, d_add, ranges
    and (at a non-zero target rate, where the counts are exact) every counter are equal; dgamma / dbeta equal the oracle's
    exact fp64 sums rounded once and the eager fp32 reductions to summation accuracy; the running buffers do not move."""
    target = 0.01 if C == 64 else 0.0
    rng = np.random.default_rng(C + 7 * relu + 3 * add + gbits)
    B, H = 8, (6 if C == 256 else 8)
    rm = torch.from_numpy((0.3 * rng.standard_normal(C)).astype(np.float32))
    rv = torch.from_numpy((0.3 + 1.5 * rng.random(C)).astype(np.float32))
    g0 = torch.from_numpy((1 + 0.3 * rng.standard_normal(C)).astype(np.float32))
    b0 = torch.from_numpy((0.2 * rng.standard_normal(C)).astype(np.float32))
    x = torch.from_numpy((rng.standard_normal((B, H, H, C)) * 1.2 + 0.3).astype(np.float32))
    a = torch.from_numpy((rng.standard_normal((B, H, H, C)) * 0.5).astype(np.float32)) if add else None
    gout = torch.from_numpy((rng.standard_normal((B, H, H, C)) * 0.7).astype(np.float32))

    ctx = O.Context(O.PhiloxNoise(SEED), exact=True)
    ol = O.BatchNorm_q(ctx, 'bn', 8, C, False, weight_decay=WD, grad_bits=gbits, target_overflow_rate=target)
    ol.layers[0].X_mean_running, ol.layers[0].X_var_running = rm.clone(), rv.clone()
    ol.layers[1].gamma.data.copy_(g0)
    ol.layers[1].beta.data.copy_(b0)
    s = ol.forward(x)
    if add:
        s = s + a
    gm = gout * (s > 0).float() if relu else gout
    y_o = torch.relu(s) if relu else s
    dx_o = ol.backward(gm)

    res = {}
    for fused in (True, False):
        rt = D.Runtime(SEED)
        pl = D.BatchNorm2d_q(8, C, weight_decay=WD, runtime=rt, fused=fused, grad_bits=gbits,
                             target_overflow_rate=target).cuda()
        rt.finalize('cuda')
        with torch.no_grad():
            for t, v in ((pl[0].X_mean_running, rm), (pl[0].X_var_running, rv), (pl[1].gamma, g0), (pl[1].beta, b0)):
                t.copy_(v)
        pl.freeze_statistics()
        assert pl.frozen and pl.training
        xin = nchw(x).contiguous(memory_format=torch.channels_last).requires_grad_(True)
        ain = nchw(a).contiguous(memory_format=torch.channels_last).requires_grad_(True) if add else None
        with launches() as seen:
            y = pl(xin, add=ain, relu=relu)
            y.backward(nchw(gout))
        torch.cuda.synchronize()
        assert (BWD in seen) == fused and (seen.count(BWD) == 1 if fused else True)
        assert not set(TRAINING_BN) & set(seen), seen
        assert torch.equal(pl[0].X_mean_running.cpu(), rm) and torch.equal(pl[0].X_var_running.cpu(), rv)
        counters = rt.flat['counters'].clone()
        rt.update_ranges()
        res[fused] = dict(y=nhwc(y), dx=nhwc(xin.grad), da=nhwc(ain.grad) if add else None, dg=pl[1].gamma.grad.cpu(),
                          db=pl[1].beta.grad.cpu(), counters=counters, ranges=list(rt.ranges().values()))
    f, e = res[True], res[False]
    for key in ('y', 'dx'):
        assert torch.equal(f[key], e[key]), (key, int((f[key] != e[key]).sum()))
    if add:
        assert torch.equal(f['da'], e['da'])
        assert torch.equal(f['da'], gm)
    if target > 0:
        assert torch.equal(f['counters'], e['counters'])
    assert f['ranges'] == e['ranges'] == [int(q.range) for q in ol.quantizers()]
    # the oracle (on the CPU): forward, and dgamma / dbeta as exact sums of the quantised products, rounded once
    assert torch.equal(f['y'], y_o), int((f['y'] != y_o).sum())
    assert torch.equal(f['dg'], ol.layers[1].dgamma.detach()), (f['dg'] - ol.layers[1].dgamma).abs().max()
    assert torch.equal(f['db'], ol.layers[1].dbeta.detach()), (f['db'] - ol.layers[1].dbeta).abs().max()
    # dx is the spec's RN(gq1 / den): the oracle's quantised gradient gq1 over the correctly rounded den, divided in fp64 and
    # rounded once.  Where the oracle's own dx differs, the channel is one where torch's CPU sqrt misrounds its den.
    den = exact_den(rv)
    gq1 = ol.layers[0].gradq
    want = torch.from_numpy((gq1.double().numpy() / den.double().numpy()).astype(np.float32))
    assert torch.equal(f['dx'], want), int((f['dx'] != want).sum())
    off = cpu_den(rv) != den
    assert torch.equal(dx_o[..., ~off], f['dx'][..., ~off])
    assert torch.equal(dx_o, (gq1 / cpu_den(rv)))
    # the eager path sums in fp32 (autograd's reductions): equal to summation accuracy, n * 2^-24 * sum |term|
    n = B * H * H
    gr, xq2 = ol.layers[1].gradq.double(), ol.layers[1].Xq.detach().double()
    bound = {'dg': (gr * xq2).abs().sum(dim=(0, 1, 2)) + (2 * WD * g0.double()).abs(), 'db': gr.abs().sum(dim=(0, 1, 2))}
    for key in ('dg', 'db'):
        err = (f[key].double() - e[key].double()).abs()
        assert bool((err <= 2 * n * 2.0 ** -24 * bound[key] + 1e-30).all()), (key, float(err.max()))


def test_frozen_batchnorm_q_in_eval_mode_is_eval_mode():
    """freeze_statistics changes nothing in eval mode: with a graph the eager path, without one the running kernels."""
    rt = D.Runtime(SEED)
    pl = D.BatchNorm2d_q(8, 16, runtime=rt).cuda()
    rt.finalize('cuda')
    seed_bn([pl], np.random.default_rng(0))
    pl.freeze_statistics().eval()
    x = torch.randn(4, 16, 6, 6, device='cuda').contiguous(memory_format=torch.channels_last).requires_grad_(True)
    with launches() as seen:
        pl(x).sum().backward()
    assert BWD not in seen and 'lbt_bn_fwd_apply_running' not in seen
    with torch.no_grad(), launches() as seen:
        pl(x)
    assert seen.count('lbt_bn_fwd_apply_running') == 1


# ---- fused units -----------------------------------------------------------------------------------------------------


def frozen_both(rt, mods, x, fn, rng):
    """fn(x) -> output, then backward of a fixed random cotangent, with frozen statistics on the fused path and with
    FUSE_UNITS off, from the same ranges, counters and step.  Asserts equal outputs, input gradients, parameter gradients,
    ranges after the controller, and unchanged running buffers; returns the fused path's launches."""
    r0, c0, s0 = rt.flat['ranges'].clone(), rt.flat['counters'].clone(), rt.dev_step.clone()
    buf0 = running_buffers(mods)
    params = [p for m in mods for p in m.parameters()]
    res, gout = [], None
    for fused in (True, False):
        rt.flat['ranges'].copy_(r0)
        rt.flat['counters'].copy_(c0)
        rt.dev_step.copy_(s0)
        for p in params:
            p.grad = None
        xin = x.detach().clone().requires_grad_(True)
        D.FUSE_UNITS = fused
        try:
            with launches() as seen:
                out = fn(xin)
                if gout is None:
                    gout = torch.from_numpy((rng.standard_normal(tuple(out.shape)) * 0.5).astype(np.float32)).cuda()
                    gout = gout.contiguous(memory_format=torch.channels_last) if out.dim() == 4 else gout
                out.backward(gout)
            torch.cuda.synchronize()
        finally:
            D.FUSE_UNITS = True
        rt.update_ranges()
        res.append((out.detach().clone(), xin.grad.clone(), [p.grad.clone() for p in params], rt.flat['ranges'].clone(), seen))
        for a, b in zip(buf0, running_buffers(mods)):
            assert torch.equal(a, b)
    (ya, dxa, ga, ra, sa), (yb, dxb, gb, rb, sb) = res
    assert torch.equal(ya, yb), int((ya != yb).sum())
    assert torch.equal(dxa, dxb), int((dxa != dxb).sum())
    for i, (p, q) in enumerate(zip(ga, gb)):
        assert torch.equal(p, q), (i, int((p != q).sum()))
    assert torch.equal(ra, rb)
    assert not set(TRAINING_BN) & set(sa), sa
    assert BWD not in sb
    return sa


def frozen_modules(rt, mods, rng):
    ml = torch.nn.ModuleList(mods).cuda()
    rt.finalize('cuda')
    seed_bn(ml.modules(), rng)
    for m in ml.modules():
        if isinstance(m, D.BatchNorm2d_q):
            m.freeze_statistics()
    return mods


def image(rng, shape, signed=True):
    x = torch.from_numpy((rng.standard_normal(shape) * 0.8).astype(np.float32))
    return (x if signed else x.abs()).cuda().contiguous(memory_format=torch.channels_last)


def test_unit_frozen_hands_mantissas_to_the_next_conv():
    rng = np.random.default_rng(1)
    rt = D.Runtime(SEED)
    conv1 = D.Conv2d_q(8, 16, 32, 3, 1, 'SAME', bias=False, input_signed=False, runtime=rt, name='c1')
    bn1 = D.BatchNorm2d_q(8, 32, relu=True, runtime=rt, name='bn1')
    conv2 = D.Conv2d_q(8, 32, 32, 3, 1, 'SAME', bias=False, input_signed=False, runtime=rt, name='c2')
    mods = frozen_modules(rt, [conv1, bn1, conv2], rng)
    hollow = []

    def fn(x):
        h = D.conv_bn_unit(conv1, bn1, x, next_conv=conv2, want_fp32=False)
        hollow.append(bool(getattr(h, '_lbt_hollow', False)))
        return conv2(h)

    seen = frozen_both(rt, mods, image(rng, (4, 16, 8, 8), signed=False), fn, rng)
    assert hollow == [True, False]           # fused: the activation between the units exists only as mantissas
    assert seen.count('lbt_bn_fwd_apply_running') == 1 and seen.count(BWD) == 1


def test_strided_block_frozen_feeds_both_consumers_and_keeps_the_block_dgrad():
    """conv+BN+ReLU producing the input of a strided basic block: the producing kernel quantises it for both consumers."""
    rng = np.random.default_rng(2)
    rt = D.Runtime(SEED)
    conv0 = D.Conv2d_q(8, 16, 16, 3, 1, 'SAME', bias=False, input_signed=True, runtime=rt, name='c0')
    bn0 = D.BatchNorm2d_q(8, 16, relu=True, runtime=rt, name='bn0')
    blk = D.ResidualBlock_q(8, 16, 32, 2, runtime=rt, name='blk')
    mods = frozen_modules(rt, [conv0, bn0, blk], rng)
    seen = frozen_both(rt, mods, image(rng, (4, 16, 16, 16)), lambda x: D.run_layers([conv0, bn0, blk], x), rng)
    assert seen.count('lbt_bn_fwd_apply_running') == 4 and seen.count(BWD) == 4


def test_bottleneck_block_frozen():
    rng = np.random.default_rng(3)
    rt = D.Runtime(SEED)
    conv0 = D.Conv2d_q(8, 16, 32, 3, 1, 'SAME', bias=False, input_signed=True, runtime=rt, name='c0')
    bn0 = D.BatchNorm2d_q(8, 32, relu=True, runtime=rt, name='bn0')
    blk = D.ResidualBottleneck_q(8, 32, 16, 2, runtime=rt, name='bott')
    mods = frozen_modules(rt, [conv0, bn0, blk], rng)
    seen = frozen_both(rt, mods, image(rng, (3, 16, 12, 12)), lambda x: D.run_layers([conv0, bn0, blk], x), rng)
    assert seen.count(BWD) == 5


@pytest.mark.parametrize('N,H', [(2, 32), (3, 36)])
def test_imagenet_stem_frozen_pooled_kernel(N, H):
    """7x7/2 conv -> BN -> ReLU -> 3x3/2 max-pool -> the next conv: the pooled running-statistics kernel forward, then the
    pool's backward and lbt_bn_bwd_running."""
    rng = np.random.default_rng(4)
    rt = D.Runtime(SEED)
    conv = D.Conv2d_q(8, 3, 64, 7, 2, 'SAME', bias=False, input_signed=True, runtime=rt, name='conv1')
    bn = D.BatchNorm2d_q(8, 64, relu=True, runtime=rt, name='conv1-bn')
    pool = D.MaxPool_q(3, 2, 'SAME')
    conv2 = D.Conv2d_q(8, 64, 64, 3, 1, 'SAME', bias=False, input_signed=False, runtime=rt, name='c2')
    mods = frozen_modules(rt, [conv, bn, conv2], rng)
    seen = frozen_both(rt, mods, image(rng, (N, 3, H, H)), lambda x: D.run_layers([conv, bn, pool, conv2], x), rng)
    assert seen.count('lbt_bn_fwd_apply_running_pooled') == 1 and 'lbt_maxpool_fwd' not in seen
    assert seen.count('lbt_maxpool_bwd') == 1 and seen.count(BWD) == 1


# ---- whole models against the exact oracle ---------------------------------------------------------------------------

IMAGE, CLASSES = 64, 100


def build(name, gbits):
    extra = dict(image=IMAGE, num_classes=CLASSES) if name.startswith('Resnet') else {}
    om = getattr(O, name)(8, weight_decay=WD, noise=O.PhiloxNoise(5), seed=1, exact=True, grad_bits=gbits, **extra)
    pm = getattr(M, name)(8, weight_decay=WD, seed=5, grad_bits=gbits, **extra).cuda()
    ov, pv = om.variables(), list(pm.parameters())
    assert len(ov) == len(pv)
    for a, b in zip(ov, pv):
        b.data.copy_(a.detach())
    return om, pm


def batch(rng, n, image, classes):
    X = torch.from_numpy((rng.standard_normal((n, image, image, 3)) * 0.5).astype(np.float32))
    y = torch.from_numpy(rng.integers(0, classes, n))
    return X, y


@pytest.mark.parametrize('name,gbits,B,image,classes', [('CIFAR10_Resnet20', None, 8, 32, 10), ('Resnet18', None, 4, IMAGE, CLASSES),
                                                       ('Resnet50', 16, 4, IMAGE, CLASSES)])
def test_frozen_training_steps_bit_exact_vs_exact_oracle(name, gbits, B, image, classes):
    """One normal training step (the running statistics move), then the statistics are frozen and three more steps run:
    after each, every gradient (dgamma / dbeta included: exact mantissa sums on both sides), weight and range equals the
    oracle's (its batch-norms set to training=False) bit for bit, and no running buffer changes.  ResNet-18's three
    downsampling blocks keep their one-launch input gradient.  Running variances whose den torch's CPU sqrt would misround
    in the oracle are moved by a few ulps, on both sides, before freezing (see cpu_den)."""
    rng = np.random.default_rng(17)
    om, pm = build(name, gbits)
    tr = Trainer(pm, lr=1e-2, momentum=0.9)
    X, y = batch(rng, B, image, classes)
    om.train_step(X, y, lr=1e-2, momentum=0.9)
    tr.step(X.permute(0, 3, 1, 2).cuda(), y.cuda())
    norms_p = [m for m in pm.modules() if isinstance(m, D.Normalization_q)]
    norms_o = oracle_bn_training(om, False)
    n_bn = len(norms_p)
    assert len(norms_o) == n_bn
    moved = 0
    for no, npm in zip(norms_o, norms_p):     # same order, and bit-identical running statistics after the normal step
        assert torch.equal(no.X_mean_running, npm.X_mean_running.cpu()) and torch.equal(no.X_var_running, npm.X_var_running.cpu())
        v, k = snap_running_var(no.X_var_running, npm.eps)
        moved += k
        no.X_var_running = v.clone()
        with torch.no_grad():
            npm.X_var_running.copy_(v)
    print('%s: %d of %d channels moved off a misrounded CPU sqrt' % (name, moved, sum(m.X_var_running.numel() for m in norms_p)))
    pm.freeze_bn_statistics()
    buf0 = running_buffers([pm])
    ovars = om.variables()
    for step in range(3):
        X, y = batch(rng, B, image, classes)
        lo = om.train_step(X, y, lr=1e-2, momentum=0.9)
        with launches() as seen:
            lp = float(tr.step(X.permute(0, 3, 1, 2).cuda(), y.cuda()))
        assert seen.count(BWD) == n_bn and not set(TRAINING_BN) & set(seen)
        if name == 'Resnet18':
            assert seen.count('lbt_conv_i8_dgrad_block') == 3
        g_o = [g for g, _ in om.grads_and_vars()]
        bad_r = [s.name for s, a, b in zip(pm.runtime.sites, om.ranges(), list(pm.ranges().values())) if a != b]
        n_g = sum(int((p.grad.cpu() != g).sum()) for p, g in zip(tr.params, g_o))
        n_w = sum(int((p.data.cpu() != v.detach()).sum()) for p, v in zip(tr.params, ovars))
        assert np.isfinite(lp) and abs(lo - lp) <= 1e-6 * max(1.0, abs(lo)), (lo, lp)
        assert not bad_r, bad_r[:8]
        assert n_g == 0 and n_w == 0, (step, n_g, n_w)
        for a, b in zip(buf0, running_buffers([pm])):
            assert torch.equal(a, b)


# ---- graph capture and the epoch loop --------------------------------------------------------------------------------


def _resnet20(seed=9):
    torch.manual_seed(3)
    pm = M.CIFAR10_Resnet20(8, weight_decay=WD, seed=seed).cuda()
    return pm, Trainer(pm, lr=1e-2, momentum=0.9)


def _state(pm, tr):
    torch.cuda.synchronize()
    return ([tr.flat_w.clone(), tr.flat_a.clone(), pm.runtime.flat['ranges'].clone(), pm.runtime.flat['counters'].clone(),
             pm.runtime.dev_step.clone()] + running_buffers([pm]))


def test_captured_frozen_step_replays_bit_identical_to_eager():
    rng = np.random.default_rng(5)
    data = [batch(rng, 16, 32, 10) for _ in range(5)]
    data = [(X.permute(0, 3, 1, 2).cuda().contiguous(memory_format=torch.channels_last), y.cuda()) for X, y in data]
    runs = []
    for graph in (False, True):
        pm, tr = _resnet20()
        tr.step(*data[0])                                  # one normal step, then frozen
        tr.freeze_bn_statistics()
        losses = []
        if graph:
            Xs, ys = data[1][0].clone(), data[1][1].clone()
            tr.capture(Xs, ys, warmup=1)                   # the warm-up step is a real (eager) frozen step
            losses.append(None)
            for X, y in data[2:]:
                Xs.copy_(X)
                ys.copy_(y)
                losses.append(float(tr.step_graph()))
            pm.freeze_bn_statistics(False)                 # toggled behind the trainer's back: the graph must not replay
            with pytest.raises(_lib.LbtError):
                tr.step_graph()
            pm.freeze_bn_statistics(True)
            tr.freeze_bn_statistics(False)                 # through the trainer: the graph is dropped
            assert not tr.captured
            with pytest.raises(_lib.LbtError, match='no step is captured'):
                tr.step_graph()
            tr.freeze_bn_statistics(True)
        else:
            losses.append(None)
            for X, y in data[1:]:
                losses.append(float(tr.step(X, y)))
            losses.pop(1)
        runs.append((losses, _state(pm, tr)))
    (la, sa), (lb, sb) = runs
    assert la == lb
    for a, b in zip(sa, sb):
        assert torch.equal(a, b)


def test_fit_freezes_at_the_requested_epoch_and_recaptures():
    rng = np.random.default_rng(4)
    X = rng.integers(0, 256, (64, 32, 32, 3), dtype=np.uint8)
    y = rng.integers(0, 10, 64)
    runs = []
    for graph in (False, True):
        pipe = PD.Pipeline(torch.from_numpy(X), torch.from_numpy(y), 'cuda', seed=2)
        pm, tr = _resnet20()
        norm = next(m for m in pm.modules() if isinstance(m, D.Normalization_q))
        modes, bufs = [], []
        capture = tr.capture

        def spy_capture(*a, **k):
            modes.append(norm.frozen)
            return capture(*a, **k)

        tr.capture = spy_capture
        buf_init = running_buffers([pm])
        test = PD.Pipeline(torch.from_numpy(X[:16]), torch.from_numpy(y[:16]), 'cuda', mean=pipe.mean, augment=False).all()
        orig_eval = tr.evaluate

        def spy_eval(*a, **k):                              # called once per epoch, after its training steps
            bufs.append(running_buffers([pm]))
            return orig_eval(*a, **k)

        tr.evaluate = spy_eval
        hist = tr.fit(pipe, 3, 32, decay_epochs=(), test=test, graph=graph, freeze_bn_epoch=1)
        assert len(hist) == 3 and all(np.isfinite(h[1]) for h in hist)
        assert all(m.frozen for m in pm.modules() if isinstance(m, D.Normalization_q))
        assert not all(torch.equal(a, b) for a, b in zip(buf_init, bufs[0]))     # epoch 0 trains the statistics
        for later in bufs[1:]:                                                     # frozen from epoch 1 on
            assert all(torch.equal(a, b) for a, b in zip(bufs[0], later))
        if graph:
            assert modes == [False, True]                   # captured in epoch 0, dropped and re-captured frozen in epoch 1
        runs.append((hist, _state(pm, tr)))
    (ha, sa), (hb, sb) = runs
    assert [h[1] for h in ha] == [h[1] for h in hb]
    for a, b in zip(sa, sb):
        assert torch.equal(a, b)


# ---- launches -------------------------------------------------------------------------------------------------------

ARITH_OPS = {'aten::add', 'aten::add_', 'aten::sub', 'aten::sub_', 'aten::rsub', 'aten::mul', 'aten::mul_', 'aten::div',
             'aten::div_', 'aten::pow', 'aten::sqrt', 'aten::mean'}


def test_frozen_step_runs_the_one_pass_backward_and_no_aten_batch_norm_arithmetic():
    """Profiler trace of a frozen ResNet-20 training step: bn_bwd_running_kernel runs, none of the training-mode BN backward
    kernels do, and the step calls no aten arithmetic a normal fused training step does not (the eager frozen path does)."""
    rng = np.random.default_rng(6)
    X, y = batch(rng, 32, 32, 10)
    X, y = X.permute(0, 3, 1, 2).cuda().contiguous(memory_format=torch.channels_last), y.cuda()

    def profile(frozen, fused=True):
        pm, tr = _resnet20()
        tr.step(X, y)
        tr.freeze_bn_statistics(frozen)
        D.FUSE_UNITS = fused
        try:
            tr.step(X, y)
            torch.cuda.synchronize()
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU,
                                                    torch.profiler.ProfilerActivity.CUDA]) as prof:
                tr.step(X, y)
                torch.cuda.synchronize()
        finally:
            D.FUSE_UNITS = True
        events = prof.events()
        ops = {}
        for e in events:
            if e.name in ARITH_OPS:
                ops[e.name] = ops.get(e.name, 0) + 1
        kernels = {e.name for e in events if e.device_type == torch.autograd.DeviceType.CUDA}
        return ops, kernels

    ops_train, k_train = profile(False)
    ops_frozen, k_frozen = profile(True)
    assert any('bn_bwd_running_kernel' in k for k in k_frozen)
    assert not any(s in k for k in k_frozen for s in ('bn_bwd1_kernel', 'bn_bwd2_kernel'))
    assert any('bn_bwd1_kernel' in k for k in k_train)
    assert all(n <= ops_train.get(op, 0) for op, n in ops_frozen.items()), (ops_frozen, ops_train)
    ops_eager, _ = profile(True, fused=False)
    assert sum(ops_eager.values()) > sum(ops_train.values())
