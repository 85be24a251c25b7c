"""Every integer contraction at the exactness bound of its s32 tensor-memory accumulator.

One accumulator may sum 65536 products exactly when at least one operand is signed (|s8*s8| <= 2^14, |u8*s8| <= 255*128),
but only 32768 when both are unsigned (|u8*u8| <= 255^2: 65536 * 65025 > 2^31 - 1).  For each entry point and operand kind
pair this file puts exactly the bound's number of products into one accumulator and checks:
  * extreme constants against an analytic reference (value * value * in-image taps, taps counted from the padding);
  * near-extreme random operands (7/8 of the entries at the extreme) against an fp64 reference on the GPU, exact below 2^53;
  * one block past the bound: launchers that split (int64 accumulation) stay exact, single-pass launchers decline with
    LBT_EUNSUPPORTED before any launch, and u8 x u8 at 65536 is declined or split.
Every case checks the kernels' error flags and, from a profiler trace, which kernel actually ran."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from lbt_b200 import _lib, gemm as G  # noqa: E402
from lbt_b200 import dfxp as D  # noqa: E402
from lbt_b200.quantizer import CNT_WORDS, MANT_S8, MANT_U8  # noqa: E402

BOUND = 65536
KIND = {'s': MANT_S8, 'u': MANT_U8}
DTYPE = {'s': torch.int8, 'u': torch.uint8}
EXTREMES = {'s': (-128, 127), 'u': (255,)}
KIND_PAIRS = ['ss', 'us', 'su', 'uu']


def _bound(kinds):
    return 32768 if kinds == 'uu' else BOUND


def _sign_pairs(kinds):
    return [(a, b) for a in EXTREMES[kinds[0]] for b in EXTREMES[kinds[1]]]


def _peak_pair(kinds):
    """The extreme pair with the largest product: the random operands sit there, so their sums stay near the bound."""
    return max(_sign_pairs(kinds), key=lambda p: abs(p[0] * p[1]))


def _near_extreme(shape, k, ext, seed):
    """`ext` in 7 of 8 entries, the rest uniform over the kind's range; generated on the GPU in row chunks."""
    gen = torch.Generator(device='cuda').manual_seed(seed)
    lo, hi = (-128, 128) if k == 's' else (0, 256)
    t = torch.full(shape, ext, dtype=DTYPE[k], device='cuda')
    rows = max(1, (1 << 26) // max(1, int(np.prod(shape[1:]))))
    for i in range(0, shape[0], rows):
        part = t[i:i + rows]
        r = torch.randint(lo, hi, part.shape, generator=gen, device='cuda', dtype=DTYPE[k])
        m = torch.randint(0, 8, part.shape, generator=gen, device='cuda', dtype=torch.uint8) == 0
        part[m] = r[m]
    return t


def _kernels(fn):
    """Run fn() under the profiler; returns its result and the names of the CUDA kernels it launched."""
    acts = [torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA]
    with torch.profiler.profile(activities=acts) as prof:
        res = fn()
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    return res, names


def _ran(names, kernel):
    return any(kernel + '<' in n or kernel + '(' in n for n in names)


def _declined(fn):
    with pytest.raises(_lib.LbtError, match=r'status -2\)'):
        fn()


def _check_gemm_errors():
    torch.cuda.synchronize()
    assert G.debug_error() == 0, 'GEMM pipeline watchdog fired'


def _check_conv_errors():
    torch.cuda.synchronize()
    assert _lib.lib().lbt_conv_debug_error() == 0
    assert _lib.lib().lbt_conv_ldg_debug_error() == 0


def _rn(x64):
    """RN_fp32 of exact fp64 values."""
    return x64.float()


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _taps_1d(n_out, n_in, k, stride, pad):
    """In-image taps of each output position along one axis: #{r < k : 0 <= o * stride + r - pad < n_in}."""
    o = np.arange(n_out)[:, None] * stride + np.arange(k)[None, :] - pad
    return ((o >= 0) & (o < n_in)).sum(1)


# ---- lbt_gemm_i8, fp32 epilogue --------------------------------------------------------------------------------------------

def _gemm_f32_case(M, N, kinds, seed):
    K = _bound(kinds)
    for a, b in _sign_pairs(kinds):
        A = torch.full((M, K), a, dtype=DTYPE[kinds[0]], device='cuda')
        B = torch.full((N, K), b, dtype=DTYPE[kinds[1]], device='cuda')
        out, names = _kernels(lambda: G.gemm_i8(A, B))
        yield out, torch.full((M, N), float(np.float32(a * b * K)), device='cuda'), names, (a, b)
        del A, B, out
    a, b = _peak_pair(kinds)
    A = _near_extreme((M, K), kinds[0], a, seed)
    B = _near_extreme((N, K), kinds[1], b, seed + 1)
    out, names = _kernels(lambda: G.gemm_i8(A, B))
    Bd = B.double()
    ref = torch.cat([_rn(A[i:i + 1024].double() @ Bd.T) for i in range(0, M, 1024)])
    yield out, ref, names, 'random'


def _gemm_f32_declines(M, N, kinds):
    K = _bound(kinds) + 16
    A = torch.zeros(M, K, dtype=DTYPE[kinds[0]], device='cuda')
    B = torch.zeros(N, K, dtype=DTYPE[kinds[1]], device='cuda')
    _declined(lambda: G.gemm_i8(A, B))
    if kinds == 'uu':
        _declined(lambda: G.gemm_i8(A[:, :BOUND], B[:, :BOUND]))


@pytest.mark.parametrize('kinds', KIND_PAIRS)
def test_gemm_f32_single_cta_at_bound(kinds):
    for out, ref, names, case in _gemm_f32_case(128, 16, kinds, 11):
        _check_gemm_errors()
        assert _ran(names, 'gemm_i8_kernel'), names
        assert torch.equal(out, ref), (case, out[0, 0].item(), ref[0, 0].item())
    _gemm_f32_declines(128, 16, kinds)


@pytest.mark.parametrize('kinds', ['ss', 'us', 'uu'])
def test_gemm_f32_cta_pair_at_bound(kinds):
    """The CTA-pair kernel takes fp32 GEMMs with N > 128 once there are at least SMs / 2 tile pairs."""
    M = 128 * (_sms() - _sms() % 2)
    try:
        _lib.lib().lbt_gemm_set_pair(1)
        for out, ref, names, case in _gemm_f32_case(M, 256, kinds, 21):
            _check_gemm_errors()
            assert _ran(names, 'gemm_i8_pair_kernel') and not _ran(names, 'gemm_i8_kernel'), names
            assert torch.equal(out, ref), (case, float((out.double() - ref.double()).abs().max()))
            del out, ref
        _gemm_f32_declines(M, 256, kinds)
    finally:
        _lib.lib().lbt_gemm_set_pair(1)


def _bnq_gemm(A, B, noise, ib, exp_const):
    M, N = A.shape[0], B.shape[0]
    counters = torch.zeros(CNT_WORDS, dtype=torch.int64, device='cuda')
    qs = _lib.QSiteStruct(bits=8, stats_minmax=1, ib=ib.data_ptr(), noise=noise.data_ptr(), seed=0, offset=0, dev_step=0,
                          counters=counters.data_ptr())
    k_out = torch.zeros(M, N, dtype=torch.int8, device='cuda')
    sums = torch.zeros(2 * N, dtype=torch.int64, device='cuda')
    G.gemm_i8(A, B, exp_const=exp_const, bnq=(qs, k_out, sums, noise.numel() // N))
    return k_out, sums


@pytest.mark.parametrize('kinds', KIND_PAIRS)
def test_gemm_fused_requantising_epilogue_at_bound(kinds):
    """k = floor(clamp(RN(exact * 2^-24) + u, -128, 127)) with explicit noise u, and the exact int64 column sums of k, k^2."""
    M, N = 128, 16
    K = _bound(kinds)
    ib = torch.tensor(7, dtype=torch.int32, device='cuda')        # 8-bit site, range 7: the mantissa scale is 2^0
    noise = torch.rand(M * N, generator=torch.Generator(device='cuda').manual_seed(3), device='cuda')
    cases = [(torch.full((M, K), a, dtype=DTYPE[kinds[0]], device='cuda'), torch.full((N, K), b, dtype=DTYPE[kinds[1]], device='cuda'))
             for a, b in _sign_pairs(kinds)]
    a, b = _peak_pair(kinds)
    cases.append((_near_extreme((M, K), kinds[0], a, 31), _near_extreme((N, K), kinds[1], b, 32)))
    for A, B in cases:
        (k_out, sums), names = _kernels(lambda: _bnq_gemm(A, B, noise, ib, -24))
        _check_gemm_errors()
        assert _ran(names, 'gemm_i8_kernel'), names
        y = _rn(A.double() @ B.double().T) * 2.0 ** -24
        k_ref = torch.floor(torch.clamp(y + noise.view(M, N), -128.0, 127.0)).to(torch.int64)
        assert torch.equal(k_out.to(torch.int64), k_ref), (A[0, 0].item(), B[0, 0].item())
        assert torch.equal(sums, torch.cat([k_ref.sum(0), (k_ref * k_ref).sum(0)]))
    A = torch.zeros(M, K + 16, dtype=DTYPE[kinds[0]], device='cuda')
    B = torch.zeros(N, K + 16, dtype=DTYPE[kinds[1]], device='cuda')
    _declined(lambda: _bnq_gemm(A, B, noise, ib, -24))
    if kinds == 'uu':
        _declined(lambda: _bnq_gemm(A[:, :BOUND], B[:, :BOUND], noise, ib, -24))


def test_gemm_fused_epilogue_statistics_flush_bound():
    """Each epilogue warp keeps int32 partials of sum k^2 over at most kBnqFlushTiles = 2048 tiles of 32 rows (2^30 for
    saturated -128 mantissas): M = 2048 tiles * 128 rows per SM, every mantissa -128, so sum k = -128 M and sum k^2 = 16384 M."""
    M, N, K = 2048 * 128 * _sms(), 16, 16
    A = torch.full((M, K), 127, dtype=torch.int8, device='cuda')
    B = torch.full((N, K), -128, dtype=torch.int8, device='cuda')
    ib = torch.tensor(7, dtype=torch.int32, device='cuda')
    noise = torch.rand(128 * N, generator=torch.Generator(device='cuda').manual_seed(4), device='cuda')
    (k_out, sums), names = _kernels(lambda: _bnq_gemm(A, B, noise, ib, 0))
    _check_gemm_errors()
    assert _ran(names, 'gemm_i8_kernel'), names
    assert bool((k_out == -128).all())
    assert sums[:N].tolist() == [-128 * M] * N and sums[N:].tolist() == [16384 * M] * N


# ---- lbt_gemm_i8, int64 split-K epilogue -----------------------------------------------------------------------------------

@pytest.mark.parametrize('kinds', KIND_PAIRS)
@pytest.mark.parametrize('alpha', [1, 65536])
def test_gemm_acc64_single_split_past_bound(kinds, alpha):
    """k_splits = 1 with K = 2 * bound + 16: the launcher must cut K into chunks the s32 accumulator sums exactly."""
    M, N = 128, 16
    K = 2 * _bound(kinds) + 16
    cases = [(torch.full((M, K), a, dtype=DTYPE[kinds[0]], device='cuda'), torch.full((N, K), b, dtype=DTYPE[kinds[1]], device='cuda'))
             for a, b in _sign_pairs(kinds)]
    a, b = _peak_pair(kinds)
    cases.append((_near_extreme((M, K), kinds[0], a, 41), _near_extreme((N, K), kinds[1], b, 42)))
    for A, B in cases:
        acc = torch.zeros(M, N, dtype=torch.int64, device='cuda')
        _, names = _kernels(lambda: G.gemm_i8_acc64(A, B, acc, alpha=alpha, k_splits=1))
        _check_gemm_errors()
        assert _ran(names, 'gemm_i8_kernel'), names
        ref = (A.double() @ B.double().T).to(torch.int64) * alpha      # |sum| < 2^33: exact in fp64
        assert torch.equal(acc, ref), (A[0, 0].item(), B[0, 0].item(), acc[0, 0].item(), ref[0, 0].item())


# ---- lbt_gemm_i8_dual: 16-bit A as byte planes (hi s8, lo u8) -------------------------------------------------------------

@pytest.mark.parametrize('b_kind', ['s', 'u'])
def test_gemm_dual_at_bound(b_kind):
    """The low-plane accumulator is u8 x B: with an unsigned B it is u8 x u8 and its bound is 32768."""
    M, N = 128, 16
    K = _bound('u' + b_kind)
    cases = []
    for hi in (-128, 127):
        for b in EXTREMES[b_kind]:
            cases.append((torch.full((M, K), hi, dtype=torch.int8, device='cuda'), torch.full((M, K), 255, dtype=torch.uint8, device='cuda'),
                          torch.full((N, K), b, dtype=DTYPE[b_kind], device='cuda')))
    cases.append((_near_extreme((M, K), 's', 127, 51), _near_extreme((M, K), 'u', 255, 52), _near_extreme((N, K), b_kind, EXTREMES[b_kind][0], 53)))
    for hi, lo, B in cases:
        out, names = _kernels(lambda: G.gemm_i8_dual(hi, lo, B))
        _check_gemm_errors()
        assert _ran(names, 'gemm_i8_kernel'), names
        ref = _rn((256 * hi.double() + lo.double()) @ B.double().T)      # |sum| < 2^15 * 2^8 * 2^16: exact in fp64
        assert torch.equal(out, ref), (hi[0, 0].item(), B[0, 0].item(), out[0, 0].item(), ref[0, 0].item())
    z = torch.zeros(M, K + 16, dtype=torch.int8, device='cuda')
    _declined(lambda: G.gemm_i8_dual(z, z.view(torch.uint8), torch.zeros(N, K + 16, dtype=DTYPE[b_kind], device='cuda')))
    if b_kind == 'u':
        z = torch.zeros(M, BOUND, dtype=torch.int8, device='cuda')
        _declined(lambda: G.gemm_i8_dual(z, z.view(torch.uint8), torch.zeros(N, BOUND, dtype=torch.uint8, device='cuda')))


# ---- gemm_i16_acc64: four byte-plane passes, the al x bl one u8 x u8 ------------------------------------------------------

@pytest.mark.parametrize('a,b', [(-1, -1), (32767, 32767), (-32767, 32767), (-32768, -32768), (32767, -32768)])
def test_gemm_i16_acc64_auto_split_one(a, b):
    """K = 65536 on a shape whose automatic split is 1 (at least one tile per SM): -1 = 256 * -1 + 255 and 32767 = 256 * 127 + 255
    put 65536 products of 255 * 255 into the low-plane pass."""
    sms, K = _sms(), BOUND
    nb = int(np.ceil(np.sqrt(sms / 2)))
    ma = -(-sms // nb)
    M, N = 128 * ma, 256 * nb
    assert ma * nb >= sms                                 # gemm_i8_acc64: k_splits = max(1, SMs // tiles) = 1
    A = torch.full((M, K), a, dtype=torch.int16, device='cuda')
    B = torch.full((N, K), b, dtype=torch.int16, device='cuda')
    calls = []
    orig = _lib.call

    def spy(fn, *args, **kw):
        calls.append((fn, args))
        return orig(fn, *args, **kw)

    _lib.call = spy
    try:
        acc, names = _kernels(lambda: G.gemm_i16_acc64(A, B))
    finally:
        _lib.call = orig
    _check_gemm_errors()
    assert _ran(names, 'gemm_i8_kernel'), names
    splits = [args[18] for fn, args in calls if fn == 'lbt_gemm_i8']
    assert splits == [1, 1, 1, 1], splits
    assert bool((acc == a * b * K).all()), (acc.min().item(), acc.max().item(), a * b * K)


# ---- convolutions ----------------------------------------------------------------------------------------------------------

def _conv_ref(src_nhwc, wp, kh, kw, sh, sw, pt, pl, OH, OW):
    """Exact fp64 implicit GEMM on the GPU: out[(n, oh, ow), co] = sum src[n, oh*sh + r - pt, ow*sw + s - pl, c] * wp[co, (r*kw + s)*C + c]."""
    N, H, W, C = src_nhwc.shape
    Cout = wp.shape[0]
    x = F.pad(src_nhwc.double().permute(0, 3, 1, 2), (pl, max((OW - 1) * sw + kw - W - pl, 0), pt, max((OH - 1) * sh + kh - H - pt, 0)))
    cols = F.unfold(x, (kh, kw), stride=(sh, sw))                        # [N, C*kh*kw, positions], rows (c, r, s)
    OHf, OWf = (x.shape[2] - kh) // sh + 1, (x.shape[3] - kw) // sw + 1
    cols = cols.view(N, C * kh * kw, OHf, OWf)[:, :, :OH, :OW].reshape(N, C * kh * kw, OH * OW)
    w = wp.double().view(Cout, kh * kw, C).permute(0, 2, 1).reshape(Cout, C * kh * kw)
    return (w @ cols).permute(0, 2, 1).reshape(N * OH * OW, Cout)


def _conv_taps(H, W, kh, kw, sh, sw, pt, pl, OH, OW):
    return torch.from_numpy(np.outer(_taps_1d(OH, H, kh, sh, pt), _taps_1d(OW, W, kw, sw, pl)).reshape(-1)).double().cuda()


def _fprop(src, sk, wp, wk, Cout, k, pad, OH, OW, out):
    N, H, W, C = src.shape
    _lib.call('lbt_conv_i8_fprop', _lib.ptr(src), KIND[sk], N, H, W, C, _lib.ptr(wp), KIND[wk], wp.stride(0), Cout, k[0], k[1], 1, 1,
              pad, pad, OH, OW, None, None, 0, None, _lib.ptr(out), Cout, None, None, None, None, _lib.stream())


@pytest.mark.parametrize('kinds', ['us', 'ss', 'uu'])
def test_conv_fprop_im2col_tma_at_bound(kinds):
    """16 x 16 filters, pad 8 on a 16 x 16 image: the centre output sums all kh*kw*C = bound products, the border ones fewer."""
    sk, wk = kinds
    C = _bound(kinds) // 256
    N, H, W, Cout, k, pad = 1, 16, 16, 16, 16, 8
    OH = OW = H + 2 * pad - k
    taps = _conv_taps(H, W, k, k, 1, 1, pad, pad, OH, OW)[:, None] * C
    assert int(taps.max()) == _bound(kinds)
    cases = [(torch.full((N, H, W, C), a, dtype=DTYPE[sk], device='cuda'), torch.full((Cout, k * k * C), b, dtype=DTYPE[wk], device='cuda'),
              (a * b * taps).expand(-1, Cout)) for a, b in _sign_pairs(kinds)]
    a, b = _peak_pair(kinds)
    x, w = _near_extreme((N, H, W, C), sk, a, 61), _near_extreme((Cout, k * k * C), wk, b, 62)
    cases.append((x, w, _conv_ref(x, w, k, k, 1, 1, pad, pad, OH, OW)))
    for x, w, ref in cases:
        out = torch.full((N * OH * OW, Cout), float('nan'), device='cuda')
        before = _lib.lib().lbt_conv_halo_launches()
        _, names = _kernels(lambda: _fprop(x, sk, w, wk, Cout, (k, k), pad, OH, OW, out))
        _check_conv_errors()
        assert _lib.lib().lbt_conv_halo_launches() == before
        assert _ran(names, 'conv_fprop_kernel'), names
        assert torch.equal(out, _rn(ref)), (x.flatten()[0].item(), w.flatten()[0].item())
    out = torch.empty(N * OH * OW, Cout, device='cuda')
    x = torch.zeros(N, H, W, C, dtype=DTYPE[sk], device='cuda')
    _declined(lambda: _fprop(x, sk, torch.zeros(Cout, 17 * k * C, dtype=DTYPE[wk], device='cuda'), wk, Cout, (17, k), pad, OH, OW, out))
    if kinds == 'uu':
        x2 = torch.zeros(N, H, W, 256, dtype=torch.uint8, device='cuda')
        _declined(lambda: _fprop(x2, 'u', torch.zeros(Cout, k * k * 256, dtype=torch.uint8, device='cuda'), 'u', Cout, (k, k), pad, OH, OW, out))


def _fprop_dual(hi, lo, wp, wk, Cout, k, pad, OH, OW, out):
    N, H, W, C = hi.shape
    _lib.call('lbt_conv_i8_fprop_dual', _lib.ptr(hi), _lib.ptr(lo), N, H, W, C, _lib.ptr(wp), KIND[wk], wp.stride(0), Cout, k[0], k[1],
              pad, pad, OH, OW, None, None, 0, _lib.ptr(out), Cout, None, _lib.stream())


@pytest.mark.parametrize('wk', ['s', 'u'])
def test_conv_fprop_dual_at_bound(wk):
    """Source as byte planes (hi s8, lo u8): with an unsigned filter the low-plane accumulator is u8 x u8 (bound 32768)."""
    C = _bound('u' + wk) // 256
    N, H, W, Cout, k, pad = 1, 16, 16, 64, 16, 8
    OH = OW = H + 2 * pad - k
    taps = _conv_taps(H, W, k, k, 1, 1, pad, pad, OH, OW)[:, None] * C
    cases = []
    for hv in (-128, 127):
        for b in EXTREMES[wk]:
            cases.append((torch.full((N, H, W, C), hv, dtype=torch.int8, device='cuda'), torch.full((N, H, W, C), 255, dtype=torch.uint8, device='cuda'),
                          torch.full((Cout, k * k * C), b, dtype=DTYPE[wk], device='cuda'), ((256 * hv + 255) * b * taps).expand(-1, Cout)))
    hi, lo = _near_extreme((N, H, W, C), 's', 127, 71), _near_extreme((N, H, W, C), 'u', 255, 72)
    w = _near_extreme((Cout, k * k * C), wk, EXTREMES[wk][0], 73)
    cases.append((hi, lo, w, _conv_ref(256 * hi.double() + lo.double(), w, k, k, 1, 1, pad, pad, OH, OW)))
    for hi, lo, w, ref in cases:
        out = torch.full((N * OH * OW, Cout), float('nan'), device='cuda')
        before = _lib.lib().lbt_conv_halo_launches()
        _, names = _kernels(lambda: _fprop_dual(hi, lo, w, wk, Cout, (k, k), pad, OH, OW, out))
        _check_conv_errors()
        assert _lib.lib().lbt_conv_halo_launches() == before
        assert _ran(names, 'conv_fprop_kernel'), names
        assert torch.equal(out, _rn(ref)), (hi.flatten()[0].item(), w.flatten()[0].item())
    out = torch.empty(N * OH * OW, Cout, device='cuda')
    z = torch.zeros(N, H, W, C, dtype=torch.int8, device='cuda')
    _declined(lambda: _fprop_dual(z, z.view(torch.uint8), torch.zeros(Cout, 17 * k * C, dtype=DTYPE[wk], device='cuda'), wk, Cout, (17, k),
                                  pad, OH, OW, out))
    if wk == 'u':
        z2 = torch.zeros(N, H, W, 256, dtype=torch.int8, device='cuda')
        _declined(lambda: _fprop_dual(z2, z2.view(torch.uint8), torch.zeros(Cout, k * k * 256, dtype=torch.uint8, device='cuda'), 'u', Cout,
                                      (k, k), pad, OH, OW, out))


def _dgrad_strided(g, gk, w2, wk, Cin, k, pad, H, W, dx):
    N, OH, OW, Cout = g.shape
    _lib.call('lbt_conv_i8_dgrad_strided', _lib.ptr(g), KIND[gk], N, OH, OW, Cout, _lib.ptr(w2), KIND[wk], w2.stride(0), Cin, k[0], k[1],
              1, 1, pad, pad, H, W, None, None, 0, _lib.ptr(dx), Cin, None, _lib.stream())


@pytest.mark.parametrize('kinds', ['us', 'ss', 'uu'])
def test_conv_dgrad_strided_at_bound(kinds):
    """Stride 1: one class, the whole 16 x 16 filter, kh*kw*Cout = bound products into the centre pixel's accumulator.  The class
    is the stride-1 correlation of g with w2 (taps in w2's order) and padding kh - 1 - pad_top."""
    gk, wk = kinds
    Cout = _bound(kinds) // 256
    N, H, W, Cin, k, pad = 1, 16, 16, 16, 16, 8
    OH = OW = 16                                         # forward geometry: 16 + 8 + 7 - 16 + 1
    p2 = k - 1 - pad
    taps = _conv_taps(OH, OW, k, k, 1, 1, p2, p2, H, W)[:, None] * Cout
    assert int(taps.max()) == _bound(kinds)
    cases = [(torch.full((N, OH, OW, Cout), a, dtype=DTYPE[gk], device='cuda'), torch.full((Cin, k * k * Cout), b, dtype=DTYPE[wk], device='cuda'),
              (a * b * taps).expand(-1, Cin)) for a, b in _sign_pairs(kinds)]
    a, b = _peak_pair(kinds)
    g, w = _near_extreme((N, OH, OW, Cout), gk, a, 81), _near_extreme((Cin, k * k * Cout), wk, b, 82)
    cases.append((g, w, _conv_ref(g, w, k, k, 1, 1, p2, p2, H, W)))
    for g, w, ref in cases:
        dx = torch.full((N * H * W, Cin), float('nan'), device='cuda')
        _, names = _kernels(lambda: _dgrad_strided(g, gk, w, wk, Cin, (k, k), pad, H, W, dx))
        _check_conv_errors()
        assert _ran(names, 'conv_fprop_kernel'), names
        assert torch.equal(dx, _rn(ref)), (g.flatten()[0].item(), w.flatten()[0].item())
    dx = torch.empty(N * H * W, Cin, device='cuda')
    z = torch.zeros(N, OH, OW, Cout, dtype=DTYPE[gk], device='cuda')
    _declined(lambda: _dgrad_strided(z, gk, torch.zeros(Cin, 17 * k * Cout, dtype=DTYPE[wk], device='cuda'), wk, Cin, (17, k), pad, H, W, dx))
    if kinds == 'uu':
        z2 = torch.zeros(N, OH, OW, 256, dtype=torch.uint8, device='cuda')
        _declined(lambda: _dgrad_strided(z2, 'u', torch.zeros(Cin, k * k * 256, dtype=torch.uint8, device='cuda'), 'u', Cin, (k, k), pad, H, W, dx))


def _dgrad_block(g, w2, gs, gsk, ws, wsk, geom, dx):
    N, OH, OW, Cout = g.shape
    Cin, k, s, pt, H, W = geom
    _, OHs, OWs, Cout_s = gs.shape
    zero = torch.zeros((), dtype=torch.int32, device='cuda')
    _lib.call('lbt_conv_i8_dgrad_block', _lib.ptr(g), MANT_S8, N, OH, OW, Cout, _lib.ptr(w2), MANT_S8, w2.stride(0), Cin, k, k, s, s,
              pt, pt, H, W, _lib.ptr(zero), _lib.ptr(zero), 0, _lib.ptr(gs), KIND[gsk], OHs, OWs, Cout_s, _lib.ptr(ws), KIND[wsk],
              ws.stride(0), _lib.ptr(zero), _lib.ptr(zero), 0, _lib.ptr(dx), Cin, None, _lib.stream())


@pytest.mark.parametrize('kinds', ['us', 'ss', 'uu'])
def test_conv_dgrad_block_shortcut_at_bound(kinds):
    """lbt_conv_i8_dgrad_block: the 1x1/2 shortcut's accumulator sums Cout_s = bound products per pixel of parity class (0, 0);
    the main 3x3/2 term (constant g = -3, w = 5) lands everywhere.  dX = RN(RN(main) + RN(shortcut)) on class (0, 0)."""
    gsk, wsk = kinds
    Cout_s = _bound(kinds)
    N, H, W, Cin, Cout, k, s = 1, 16, 16, 64, 128, 3, 2
    OH, pt, _ = D.same_pad(H, k, s)
    geom = (Cin, k, s, pt, H, W)
    OHs = OWs = H // 2
    gv, wv = -3, 5
    g = torch.full((N, OH, OH, Cout), gv, dtype=torch.int8, device='cuda')
    w2 = torch.full((Cin, k * k * Cout), wv, dtype=torch.int8, device='cuda')
    pos = (np.arange(OH)[:, None] * s + np.arange(k)[None, :] - pt).ravel()
    th = torch.from_numpy(np.bincount(pos[(pos >= 0) & (pos < H)], minlength=H))   # taps (oh, r) that reach input row y
    main = _rn((gv * wv * Cout * torch.outer(th, th)).double().cuda())[None, :, :, None].expand(N, H, W, Cin).contiguous()
    cases = [(torch.full((N, OHs, OWs, Cout_s), a, dtype=DTYPE[gsk], device='cuda'),
              torch.full((Cin, Cout_s), b, dtype=DTYPE[wsk], device='cuda')) for a, b in _sign_pairs(kinds)]
    a, b = _peak_pair(kinds)
    cases.append((_near_extreme((N, OHs, OWs, Cout_s), gsk, a, 91), _near_extreme((Cin, Cout_s), wsk, b, 92)))
    for gs, ws in cases:
        dx = torch.full((N, H, W, Cin), float('nan'), device='cuda')
        _, names = _kernels(lambda: _dgrad_block(g, w2, gs, gsk, ws, wsk, geom, dx))
        _check_conv_errors()
        assert _ran(names, 'conv_dgrad_block_kernel'), names
        short = _rn(gs.double().reshape(-1, Cout_s) @ ws.double().T).view(N, OHs, OWs, Cin)   # |sum| < 2^32: exact in fp64
        want = main.clone()
        want[:, ::2, ::2] = main[:, ::2, ::2] + short
        assert torch.equal(dx, want), (gs.flatten()[0].item(), ws.flatten()[0].item())
    dx = torch.empty(N, H, W, Cin, device='cuda')
    gs = torch.zeros(N, OHs, OWs, Cout_s + 128, dtype=DTYPE[gsk], device='cuda')
    _declined(lambda: _dgrad_block(g, w2, gs, gsk, torch.zeros(Cin, Cout_s + 128, dtype=DTYPE[wsk], device='cuda'), wsk, geom, dx))
    if kinds == 'uu':
        gs = torch.zeros(N, OHs, OWs, BOUND, dtype=torch.uint8, device='cuda')
        _declined(lambda: _dgrad_block(g, w2, gs, 'u', torch.zeros(Cin, BOUND, dtype=torch.uint8, device='cuda'), 'u', geom, dx))


# ---- weight gradients (int64 accumulation: the launchers split the pixels, never decline) ----------------------------------

def _wgrad(x, xk, g, gk, Cout, k, pad, OH, OW, acc, k_splits, g_lo=None):
    N, H, W, C = x.shape
    if g_lo is None:
        _lib.call('lbt_conv_i8_wgrad', _lib.ptr(x), KIND[xk], N, H, W, C, _lib.ptr(g), KIND[gk], Cout, k, k, 1, 1, pad, pad, OH, OW,
                  _lib.ptr(acc), 1, k_splits, _lib.stream())
    else:
        _lib.call('lbt_conv_i8_wgrad_dual', _lib.ptr(x), KIND[xk], N, H, W, C, _lib.ptr(g), _lib.ptr(g_lo), Cout, k, k, 1, 1, pad, pad,
                  OH, OW, _lib.ptr(acc), 1, k_splits, _lib.stream())


def _wgrad_ref(x, g, k, pad, chunk):
    """dW[(r, s, c), co] = sum over pixels of x[n, oh + r - pad, ow + s - pad, c] * g[(n, oh, ow), co] in fp64 (exact), images
    in chunks."""
    N, H, W, C = x.shape
    Cout = g.shape[-1]
    g = g.view(N, H * W, Cout)
    ref = torch.zeros(C * k * k, Cout, dtype=torch.float64, device='cuda')
    for i in range(0, N, chunk):
        xc = F.pad(x[i:i + chunk].double().permute(0, 3, 1, 2), (pad,) * 4)
        cols = F.unfold(xc, (k, k))                                        # [n, C*k*k, H*W]
        ref += (cols @ g[i:i + chunk].double()).sum(0)
    return ref.view(C, k * k, Cout).permute(1, 0, 2).reshape(k * k * C, Cout)


def _wgrad_taps(H, W, k, pad):
    t = np.outer(_taps_1d(k, H, H, 1, pad), _taps_1d(k, W, W, 1, pad))     # tap (r, s): output pixels whose tap is in the image
    return torch.from_numpy(t.reshape(-1)).double().cuda()


def _wgrad_cases(shape, kinds, C, Cout, seed, dual=False):
    """(x, g, g_lo, reference) for every extreme pair and one near-extreme random draw; dual: g is the high plane (s8) of
    256 * hi + 255."""
    N, H, W = shape
    k, pad = 3, 1
    taps = _wgrad_taps(H, W, k, pad).repeat_interleave(C)[:, None] * N
    gk = 's' if dual else kinds[1]
    for a, b in _sign_pairs(kinds[0] + gk):
        x = torch.full((N, H, W, C), a, dtype=DTYPE[kinds[0]], device='cuda')
        g = torch.full((N * H * W, Cout), b, dtype=DTYPE[gk], device='cuda')
        lo = torch.full((N * H * W, Cout), 255, dtype=torch.uint8, device='cuda') if dual else None
        yield x, g, lo, (a * ((256 * b + 255) if dual else b) * taps).expand(-1, Cout)
    a, b = _peak_pair(kinds[0] + gk)
    x = _near_extreme((N, H, W, C), kinds[0], a, seed)
    g = _near_extreme((N * H * W, Cout), gk, b, seed + 1)
    lo = _near_extreme((N * H * W, Cout), 'u', 255, seed + 2) if dual else None
    gv = 256 * g.double() + lo.double() if dual else g
    yield x, g, lo, _wgrad_ref(x, gv, k, pad, max(1, 65536 // (H * W)))


@pytest.mark.parametrize('kinds', KIND_PAIRS)
@pytest.mark.parametrize('past', [False, True])
def test_conv_wgrad_tma_single_split(kinds, past):
    """lbt_conv_i8_wgrad, k_splits = 1, C = 64: 65536 pixels (512 blocks: u8 x u8 must split them) or one block more."""
    shape = (1, 128, 513) if past else (1, 256, 256)
    C = Cout = 64
    for x, g, _, ref in _wgrad_cases(shape, kinds, C, Cout, 101):
        acc = torch.zeros(9 * C, Cout, dtype=torch.int64, device='cuda')
        _, names = _kernels(lambda: _wgrad(x, kinds[0], g, kinds[1], Cout, 3, 1, shape[1], shape[2], acc, 1))
        _check_conv_errors()
        assert _ran(names, 'conv_wgrad_kernel'), names
        assert torch.equal(acc, ref.to(torch.int64)), (x.flatten()[0].item(), g.flatten()[0].item())


@pytest.mark.parametrize('xk', ['u', 's'])
def test_conv_wgrad_dual_single_split(xk):
    """lbt_conv_i8_wgrad_dual, k_splits = 1, 65536 pixels: x x g_lo is u8 x u8 for an unsigned source."""
    shape = (1, 256, 256)
    C = Cout = 64
    for x, hi, lo, ref in _wgrad_cases(shape, xk + 'u', C, Cout, 111, dual=True):
        acc = torch.zeros(9 * C, Cout, dtype=torch.int64, device='cuda')
        _, names = _kernels(lambda: _wgrad(x, xk, hi, 's', Cout, 3, 1, shape[1], shape[2], acc, 1, g_lo=lo))
        _check_conv_errors()
        assert _ran(names, 'conv_wgrad_kernel'), names
        assert torch.equal(acc, ref.to(torch.int64)), (x.flatten()[0].item(), hi.flatten()[0].item())


@pytest.mark.parametrize('kinds', KIND_PAIRS)
def test_conv_wgrad_gather_many_blocks_per_cta(kinds, record_property):
    """C = Cout = 16, automatic split: the cp.async-gather kernel spreads the pixels over all SMs (two CTAs each), 300 pixel
    blocks per CTA — above the 256 that u8 x u8 allows, so that pair must fall back to the TMA kernel.  Passes on either
    kernel; the one that ran is recorded."""
    N, H, W = 2 * _sms() * 300 * 128 // (64 * 64), 64, 64
    C = Cout = 16
    for x, g, _, ref in _wgrad_cases((N, H, W), kinds, C, Cout, 121):
        acc = torch.zeros(9 * C, Cout, dtype=torch.int64, device='cuda')
        _, names = _kernels(lambda: _wgrad(x, kinds[0], g, kinds[1], Cout, 3, 1, H, W, acc, 0))
        _check_conv_errors()
        gather, tma = _ran(names, 'conv_wgrad_ldg_kernel'), _ran(names, 'conv_wgrad_kernel')
        assert gather != tma, names
        record_property('kernel', 'gather' if gather else 'tma')
        assert torch.equal(acc, ref.to(torch.int64)), (x.flatten()[0].item(), g.flatten()[0].item())
        if kinds == 'uu':
            assert tma, names
        del x, g, ref
