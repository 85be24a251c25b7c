"""Fused Conv2d_q + BatchNorm2d_q units (tensor-core epilogue re-quantisation, mantissa hand-offs between
modules) against the same modules run one after the other: identical quantiser ids, ranges, noise streams and
arithmetic, so every result must be BIT-identical."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from lbt_b200 import dfxp as D, models as M  # noqa: E402
from lbt_b200.trainer import Trainer  # noqa: E402


def _run(name, fused, steps, batch, image, kw):
    D.FUSE_UNITS = fused
    try:
        torch.manual_seed(3)
        model = getattr(M, name)(8, weight_decay=2e-4, seed=9, **kw).cuda()
        tr = Trainer(model, lr=1e-2, momentum=0.9)
        rng = np.random.default_rng(1)
        losses = []
        for _ in range(steps):
            X = torch.from_numpy((rng.standard_normal((batch, image, image, 3)) * 0.5).astype(np.float32)).cuda()
            y = torch.from_numpy(rng.integers(0, 10, batch)).cuda()
            losses.append(float(tr.step(X.permute(0, 3, 1, 2), y)))
        torch.cuda.synchronize()
        return dict(losses=losses, w=tr.flat_w.clone(), g=tr.flat_g.clone(), a=tr.flat_a.clone(),
                    ranges=model.runtime.flat['ranges'].clone(), counters=model.runtime.flat['counters'].clone(),
                    bn=[b.clone() for n, b in model.named_buffers() if 'running' in n])
    finally:
        D.FUSE_UNITS = True


@pytest.mark.parametrize('name,batch,image,kw', [
    ('CIFAR10_Resnet20', 16, 32, {}),
    ('CIFAR10_Resnet20', 5, 32, {}),                                  # ragged M tiles (5*32*32 = 40 tiles; 5*8*8 = 2.5 tiles)
    ('Resnet18', 4, 64, dict(image=64, num_classes=10)),              # stride-2 units, max-pool after the stem, 128..512 channels
    ('Resnet50', 2, 64, dict(image=64, num_classes=10)),              # bottlenecks: 1x1 units through lbt_gemm_i8
])
def test_fused_units_equal_unfused_bit_for_bit(name, batch, image, kw):
    a = _run(name, True, 3, batch, image, kw)
    b = _run(name, False, 3, batch, image, kw)
    assert a['losses'] == b['losses'], (a['losses'], b['losses'])
    assert torch.equal(a['ranges'], b['ranges'])
    assert torch.equal(a['counters'], b['counters'])
    for k in ('g', 'w', 'a'):
        assert torch.equal(a[k].view(torch.int32), b[k].view(torch.int32)), k
    for x, y in zip(a['bn'], b['bn']):
        assert torch.equal(x, y)


def test_fused_unit_hands_mantissas_to_the_next_conv():
    """Inside a residual block the activation between bn1 and conv2 exists only as mantissas."""
    torch.manual_seed(0)
    rt = D.Runtime(1)
    blk = D.ResidualBlock_q(8, 16, 16, 1, runtime=rt).cuda()
    x = torch.rand(4, 16, 8, 8, device='cuda').contiguous(memory_format=torch.channels_last)
    seen = {}
    orig = D._conv_quantize_input

    def spy(layer, t, geom):
        seen[layer.name] = (getattr(t, '_lbt_hollow', False), id(layer.qX) in (getattr(t, '_lbt_q', None) or {}))
        return orig(layer, t, geom)

    D._conv_quantize_input = spy
    try:
        y = blk(x)
    finally:
        D._conv_quantize_input = orig
    assert seen['block-2'] == (True, True)          # conv2 consumed bn1's fused mantissas, no fp32 tensor
    assert seen['block-1'] == (False, False)
    assert y.shape == x.shape and bool(torch.isfinite(y).all())


@pytest.mark.parametrize('N,C,H,W,k,s,padding', [(3, 8, 9, 7, 3, 2, 'SAME'), (2, 64, 32, 32, 3, 2, 'SAME'),
                                                 (2, 16, 8, 8, 2, 2, 'VALID'), (1, 4, 5, 5, 3, 1, 'SAME'), (2, 12, 11, 13, 5, 3, 'SAME')])
def test_maxpool_kernels_equal_torch(N, C, H, W, k, s, padding):
    """lbt_maxpool_fwd/bwd vs -inf padding + torch max_pool2d (the oracle's restatement of tf.nn.max_pool), with exact
    ties (post-ReLU zeros): forward and gradient bit-identical."""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(N * 100 + C)
    x = torch.relu(torch.randn(N, C, H, W, generator=g)).mul(4).round().div(4)         # many ties, many zeros
    pool = D.MaxPool_q(k, s, padding)
    xa = x.cuda().contiguous(memory_format=torch.channels_last).requires_grad_(True)
    ya = pool(xa)
    xb = x.clone().requires_grad_(True)
    if padding == 'SAME':
        _, pt, pb = D.same_pad(H, k, s)
        _, pl, pr = D.same_pad(W, k, s)
        xp = F.pad(xb, (pl, pr, pt, pb), value=float('-inf'))
    else:
        xp = xb
    yb = F.max_pool2d(xp, k, s)
    assert ya.shape == yb.shape
    assert torch.equal(ya.cpu(), yb)
    go = torch.randn(yb.shape, generator=g)
    ya.backward(go.cuda())
    yb.backward(go)
    assert torch.equal(xa.grad.cpu(), xb.grad)


def test_avgpool_and_xent_kernels_match_torch():
    """lbt_avgpool_* bit-identical to torch's avg_pool2d (the oracle's restatement of tf.nn.avg_pool); the softmax
    cross-entropy within fp32 round-off of torch's (different exp/log implementations)."""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(3)
    for (N, C, H, k, s) in [(5, 64, 8, 8, 1), (3, 16, 9, 3, 2), (2, 8, 7, 2, 2)]:
        x = torch.randn(N, C, H, H, generator=g)
        xa = x.cuda().contiguous(memory_format=torch.channels_last).requires_grad_(True)
        ya = D.AvgPool_q(k, s)(xa)
        xb = x.clone().requires_grad_(True)
        yb = F.avg_pool2d(xb, k, s)
        assert torch.equal(ya.cpu(), yb)
        go = torch.randn(yb.shape, generator=g)
        ya.backward(go.cuda())
        yb.backward(go)
        assert torch.equal(xa.grad.cpu(), xb.grad)
    for (B, C) in [(256, 10), (7, 1000), (1, 3)]:
        z = torch.randn(B, C, generator=g) * 3
        y = torch.randint(0, C, (B,), generator=g)
        za = z.cuda().requires_grad_(True)
        la = D.softmax_cross_entropy(za, y.cuda())
        zb = z.clone().requires_grad_(True)
        lb = F.cross_entropy(zb, y)
        la.backward()
        lb.backward()
        assert abs(float(la) - float(lb)) <= 1e-6 * max(1.0, abs(float(lb)))
        assert float((za.grad.cpu() - zb.grad).abs().max()) <= 1e-7


def test_xent_cluster_kernel_same_bits_as_single_cta_order():
    """The 8-CTA cluster version of lbt_softmax_xent_fwd (B > 32 and B*C > 8192, e.g. ImageNet's 256 x 1000) adds the row losses
    in the single-CTA kernel's order: rows are independent, so the row losses come from B=1 calls (loss = 0.0f + l), warp w
    sums rows w, w+32, ... from 0.0f, then the 32 partials in order, then / B — all in fp32."""
    import numpy as np
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(11)
    for (B, C) in [(256, 1000), (77, 300), (4096, 10)]:
        z = (torch.randn(B, C, generator=g) * 3).cuda()
        y = torch.randint(0, C, (B,), generator=g).cuda()
        la = D.softmax_cross_entropy(z, y)
        rows = None
        if B <= 256:
            rows = np.array([float(D.softmax_cross_entropy(z[i:i + 1], y[i:i + 1])) for i in range(B)], dtype=np.float32)
        lb = F.cross_entropy(z.cpu(), y.cpu())
        assert abs(float(la) - float(lb)) <= 2e-6 * max(1.0, abs(float(lb)))
        if rows is None:
            continue
        parts = np.zeros(32, dtype=np.float32)
        for w in range(32):
            p = np.float32(0.0)
            for r in range(w, B, 32):
                p = np.float32(p + rows[r])
            parts[w] = p
        t = np.float32(0.0)
        for w in range(32):
            t = np.float32(t + parts[w])
        assert np.float32(float(la)).tobytes() == np.float32(t / np.float32(B)).tobytes()


@pytest.mark.parametrize('name,batch,image,kw', [('Resnet18', 4, 64, dict(image=64, num_classes=10)),
                                                 ('Resnet18', 3, 60, dict(image=60, num_classes=10)),      # 30 x 30 -> 15 x 15: ragged tiles and windows
                                                 ('Resnet18', 5, 96, dict(image=96, num_classes=10)),      # 48 x 48: several tiles per image, halo between them
                                                 ('Resnet50', 2, 64, dict(image=64, num_classes=10, grad_bits=16))])
def test_bn_apply_with_pool_folded_in_equals_two_kernels(name, batch, image, kw):
    """lbt_bn_fwd_apply_pooled (BN pass 2 + ReLU + the stem's 3x3/2 max-pool in one kernel, no fp32 module output) vs
    lbt_bn_fwd_apply + lbt_maxpool_fwd: losses, gradients, weights, momentum, ranges, counters and running statistics of three
    training steps bit-identical."""
    from lbt_b200 import _lib
    seen = []
    orig = _lib.try_call

    def spy(fn, *a, **k):
        ok = orig(fn, *a, **k)
        seen.append((fn, ok))
        return ok

    res = {}
    for on in (True, False):
        D.FUSE_POOL_FWD = on
        del seen[:]
        _lib.try_call = spy
        try:
            res[on] = _run(name, True, 3, batch, image, kw)
        finally:
            _lib.try_call = orig
            D.FUSE_POOL_FWD = True
        n = sum(1 for fn, ok in seen if fn == 'lbt_bn_fwd_apply_pooled' and ok)
        assert n == (3 if on else 0), (on, n)
    a, b = res[True], res[False]
    assert a['losses'] == b['losses'], (a['losses'], b['losses'])
    assert torch.equal(a['ranges'], b['ranges'])
    assert torch.equal(a['counters'], b['counters'])
    for k in ('g', 'w', 'a'):
        assert torch.equal(a[k].view(torch.int32), b[k].view(torch.int32)), k
    for x, y in zip(a['bn'], b['bn']):
        assert torch.equal(x, y)
