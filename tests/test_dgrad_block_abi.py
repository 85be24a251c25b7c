"""CPU-side checks of lbt_conv_i8_dgrad_block: bad arguments are rejected before any CUDA call, so these run without a GPU."""
import ctypes

from lbt_b200 import _lib

S8, U8 = 1, 2


def _bufs():
    f = (ctypes.c_float * 64)()
    p = ctypes.cast(f, ctypes.c_void_p)
    ib = ctypes.cast((ctypes.c_int32 * 1)(2), ctypes.c_void_p)
    return p, ib


def _call(g=True, g_kind=S8, N=2, OH=14, OW=14, Cout=128, w2=True, ldw=9 * 128, Cin=64, kh=3, kw=3, sh=2, sw=2, pt=0, pl=0, H=28, W=28,
          gs=True, gs_kind=S8, OHs=14, OWs=14, Cout_s=128, ws=True, ldws=128, dx=True, ldc=64, addend=False, ib=True):
    h = _lib.lib()
    p, ibp = _bufs()
    i = ibp if ib else None
    return h.lbt_conv_i8_dgrad_block(p if g else None, g_kind, N, OH, OW, Cout, p if w2 else None, S8, ldw, Cin, kh, kw, sh, sw, pt, pl,
                                     H, W, i, i, -14, p if gs else None, gs_kind, OHs, OWs, Cout_s, p if ws else None, S8, ldws, i, i,
                                     -14, p if dx else None, ldc, p if addend else None, None)


def test_dgrad_block_is_declared_and_bound():
    assert 'lbt_conv_i8_dgrad_block' in _lib.SIGNATURES
    assert hasattr(_lib.lib(), 'lbt_conv_i8_dgrad_block')


def test_dgrad_block_rejects_bad_arguments_without_gpu():
    EINVAL, EUNSUP = -1, -2
    assert _call(g=False) == EINVAL
    assert _call(w2=False) == EINVAL
    assert _call(dx=False) == EINVAL
    assert _call(ib=False) == EINVAL
    assert _call(g_kind=7) == EINVAL
    assert _call(N=0) == EINVAL
    assert _call(Cin=-4) == EINVAL
    assert _call(pt=-1) == EINVAL
    assert _call(ldc=32) == EINVAL                    # row pitch below Cin
    assert _call(ldw=128) == EINVAL                   # row pitch below kh * kw * Cout
    assert _call(ws=False) == EINVAL                  # a shortcut gradient without its filter
    assert _call(gs_kind=9) == EINVAL
    assert _call(ldws=64) == EINVAL
    assert _call(Cin=66, ldc=68) == EUNSUP            # Cin % 4 != 0
    assert _call(Cin=96, ldc=96) == EUNSUP            # neither 64 nor a multiple of 128
    assert _call(sh=3, sw=3) == EUNSUP                # strides above 2
    assert _call(Cout=48, ldw=9 * 48) == EUNSUP       # channel chunk of g
    assert _call(Cout_s=64, ldws=64) == EUNSUP        # the shortcut's channel chunk differs from g's
    assert _call(OHs=13) == EUNSUP                    # the shortcut does not sample parity class (0, 0)
    assert _call(OWs=15) == EUNSUP
    assert _call(addend=True) == EUNSUP               # shortcut and external addend together
    assert _call(ldc=66) == EUNSUP                    # misaligned rows of dX
