"""lbt_conv_i8_dgrad_block (a downsampling block's whole input gradient in one launch: every parity class of the strided
convolution and the 1x1 shortcut in a second accumulator) against the two lbt_conv_i8_dgrad_strided launches it replaces
and against the exact transposed convolutions in fp64; training steps with FUSE_BLOCK_DGRAD on and off.  All comparisons
are exact (torch.equal)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from lbt_b200 import _lib, dfxp as D, models as M, quantizer as Q  # noqa: E402
from lbt_b200.trainer import Trainer  # noqa: E402


def _ptr(t):
    return _lib.ptr(t)


def _exact_dgrad(gm, wm, s, pt, pl, H, W):
    """fp64 transposed convolution of g [N, OH, OW, Cout] with W [kh, kw, Cin, Cout], 'SAME' offsets (pt, pl): [N, H, W, Cin]."""
    N = gm.shape[0]
    Cin = wm.shape[2]
    full = F.conv_transpose2d(gm.double().permute(0, 3, 1, 2), wm.double().permute(3, 2, 0, 1), stride=s)
    ref = torch.zeros(N, Cin, H, W, dtype=torch.float64, device='cuda')
    hh, ww = min(H, full.shape[2] - pt), min(W, full.shape[3] - pl)
    ref[:, :, :hh, :ww] = full[:, :, pt:pt + hh, pl:pl + ww]
    return ref.permute(0, 2, 3, 1)


SHAPES = [
    # N, H, W, Cin, Cout, k, shortcut, addend
    (2, 56, 56, 64, 128, 3, True, False),      # ResNet-18 stage 2
    (2, 28, 28, 128, 256, 3, True, False),     # stage 3
    (2, 14, 14, 256, 512, 3, True, False),     # stage 4
    (3, 27, 31, 64, 128, 3, True, False),      # odd image
    (2, 28, 28, 128, 256, 3, False, False),    # no shortcut
    (2, 28, 28, 128, 256, 3, False, True),     # no shortcut, external addend
    (2, 28, 28, 128, 256, 1, True, False),     # 1x1/2 main convolution (bottleneck-like): three tap-less classes
    (2, 27, 31, 64, 128, 1, False, True),      # 1x1/2, tap-less classes get the addend
    (2, 27, 31, 64, 128, 1, False, False),     # 1x1/2, tap-less classes get zeros
]


@pytest.mark.parametrize('N,H,W,Cin,Cout,k,shortcut,with_addend', SHAPES)
def test_dgrad_block_equals_two_strided_calls_and_exact(N, H, W, Cin, Cout, k, shortcut, with_addend):
    s = 2
    rng = np.random.default_rng(N * H + W + Cin + k)
    OH, pt, _ = D.same_pad(H, k, s)
    OW, pl, _ = D.same_pad(W, k, s)
    OHs, OWs = -(-H // s), -(-W // s)
    wm = torch.from_numpy(rng.integers(-128, 128, (k, k, Cin, Cout), dtype=np.int8)).cuda()
    gm = torch.from_numpy(rng.integers(-128, 128, (N, OH, OW, Cout), dtype=np.int8)).cuda()
    wsm = torch.from_numpy(rng.integers(-128, 128, (1, 1, Cin, Cout), dtype=np.int8)).cuda()
    gsm = torch.from_numpy(rng.integers(-128, 128, (N, OHs, OWs, Cout), dtype=np.int8)).cuda()
    ib = torch.tensor([3, -2, 1, 0], dtype=torch.int32, device='cuda')   # ranges of g, W, g_short, W_short
    e, es = -14, -13
    perm = torch.tensor(D._class_perm(k, k, s, s), device='cuda')
    w2 = wm.view(k * k, Cin, Cout).index_select(0, perm).permute(1, 0, 2).reshape(Cin, k * k * Cout).contiguous()
    ws2 = wsm.view(Cin, Cout).contiguous()
    addend = torch.randn(N, H, W, Cin, device='cuda') if with_addend else None
    S8 = Q.MANT_S8

    def strided(g, w, kk, p_t, p_l, oh, ow, ib_g, ib_w, ex, out, ad):
        _lib.call('lbt_conv_i8_dgrad_strided', _ptr(g), S8, N, oh, ow, Cout, _ptr(w), S8, w.stride(0), Cin, kk, kk, s, s, p_t, p_l,
                  H, W, _ptr(ib_g), _ptr(ib_w), ex, _ptr(out), Cin, _ptr(ad), _lib.stream())

    # the sequence the block kernel replaces
    ref = torch.empty(N, H, W, Cin, device='cuda')
    ad = addend
    if shortcut:
        ad = torch.empty(N, H, W, Cin, device='cuda')
        strided(gsm, ws2, 1, 0, 0, OHs, OWs, ib[2:3], ib[3:4], es, ad, None)
    strided(gm, w2, k, pt, pl, OH, OW, ib[0:1], ib[1:2], e, ref, ad)

    got = torch.full((N, H, W, Cin), float('nan'), device='cuda')
    _lib.call('lbt_conv_i8_dgrad_block', _ptr(gm), S8, N, OH, OW, Cout, _ptr(w2), S8, w2.stride(0), Cin, k, k, s, s, pt, pl, H, W,
              _ptr(ib[0:1]), _ptr(ib[1:2]), e, _ptr(gsm) if shortcut else None, S8, OHs, OWs, Cout, _ptr(ws2) if shortcut else None,
              S8, ws2.stride(0), _ptr(ib[2:3]), _ptr(ib[3:4]), es, _ptr(got), Cin, _ptr(addend), _lib.stream())
    torch.cuda.synchronize()
    assert _lib.lib().lbt_conv_debug_error() == 0
    assert torch.equal(got, ref), int((got != ref).sum())

    want = (_exact_dgrad(gm, wm, s, pt, pl, H, W) * 2.0 ** (3 - 2 + e)).float()
    if shortcut:
        want = want + (_exact_dgrad(gsm, wsm, s, 0, 0, H, W) * 2.0 ** (1 + 0 + es)).float()
    if addend is not None:
        want = want + addend
    assert torch.equal(got, want.contiguous())


# ---- training steps -------------------------------------------------------------------------------------------------


def _spy():
    seen = []
    orig_call, orig_try = _lib.call, _lib.try_call

    def call(fn, *a, **k):
        seen.append(fn)
        return orig_call(fn, *a, **k)

    def try_call(fn, *a, **k):
        ok = orig_try(fn, *a, **k)
        if ok:
            seen.append(fn)
        return ok

    _lib.call, _lib.try_call = call, try_call
    return seen, (orig_call, orig_try)


def _unspy(orig):
    _lib.call, _lib.try_call = orig


def _run(name, fused, steps, batch, image, kw, graph=False):
    D.FUSE_BLOCK_DGRAD = fused
    try:
        torch.manual_seed(3)
        model = getattr(M, name)(8, weight_decay=2e-4, seed=9, **kw).cuda()
        tr = Trainer(model, lr=1e-2, momentum=0.9)
        rng = np.random.default_rng(1)

        def data():
            X = torch.from_numpy((rng.standard_normal((batch, image, image, 3)) * 0.5).astype(np.float32)).cuda()
            y = torch.from_numpy(rng.integers(0, 10, batch)).cuda()
            return X.permute(0, 3, 1, 2), y

        losses = []
        if graph:
            Xs, ys = data()
            Xs = Xs.contiguous(memory_format=torch.channels_last)
            tr.capture(Xs, ys, warmup=1)
            for _ in range(steps - 1):
                X, y = data()
                Xs.copy_(X)
                ys.copy_(y)
                losses.append(float(tr.step_graph()))
        else:
            for _ in range(steps):
                X, y = data()
                losses.append(float(tr.step(X, y)))
        torch.cuda.synchronize()
        assert _lib.lib().lbt_conv_debug_error() == 0
        return dict(losses=losses, w=tr.flat_w.clone(), g=tr.flat_g.clone(), a=tr.flat_a.clone(),
                    ranges=model.runtime.flat['ranges'].clone(), counters=model.runtime.flat['counters'].clone(),
                    bn=[b.clone() for n, b in model.named_buffers() if 'running' in n])
    finally:
        D.FUSE_BLOCK_DGRAD = True


def _assert_same(a, b):
    assert a['losses'] == b['losses']
    for key in ('w', 'g', 'a', 'ranges', 'counters'):
        assert torch.equal(a[key], b[key]), key
    assert all(torch.equal(x, y) for x, y in zip(a['bn'], b['bn']))


@pytest.mark.parametrize('name,batch,image,graph', [('Resnet18', 4, 64, False), ('Resnet18', 3, 60, False), ('Resnet18', 4, 64, True),
                                                    ('Resnet50', 2, 64, False), ('Resnet50', 2, 64, True)])
def test_training_steps_equal_with_and_without_block_dgrad(name, batch, image, graph):
    kw = dict(image=image, num_classes=10)
    on = _run(name, True, 3, batch, image, kw, graph)
    off = _run(name, False, 3, batch, image, kw, graph)
    _assert_same(on, off)


def test_resnet18_step_issues_three_block_dgrads_and_no_strided_dgrad():
    seen, orig = _spy()
    D._block_dgrad_count = 0
    try:
        _run('Resnet18', True, 1, 4, 64, dict(image=64, num_classes=10))
    finally:
        _unspy(orig)
    assert seen.count('lbt_conv_i8_dgrad_block') == 3, seen
    assert D._block_dgrad_count == 3
    assert 'lbt_conv_i8_dgrad_strided' not in seen
    seen, orig = _spy()
    try:
        _run('Resnet18', False, 1, 4, 64, dict(image=64, num_classes=10))
    finally:
        _unspy(orig)
    assert 'lbt_conv_i8_dgrad_block' not in seen and seen.count('lbt_conv_i8_dgrad_strided') == 6
