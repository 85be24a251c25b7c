"""CPU-side checks of the frozen-statistics batch-norm backward entry point (lbt_bn_bwd_running): bad arguments are rejected
with LBT_EINVAL before any CUDA call, so these run without a GPU."""
import ctypes

from lbt_b200 import _lib
from lbt_b200.quantizer import MANT_S16 as S16, MANT_S8 as S8


def _bufs():
    f = (ctypes.c_float * 64)()
    p = ctypes.cast(f, ctypes.c_void_p)
    ib = ctypes.cast((ctypes.c_int32 * 1)(2), ctypes.c_void_p)
    return p, ib


def _bwd(g=True, k2=True, gq=True, bq=True, run_var=True, sums=True, C=8, relu=1, out=None, dx=True, q_grad=None, gm=None,
         gm_lo=None, bits2=8, bits_g2=8, bits_g1=8, kind=S8, ib_g=True):
    h = _lib.lib()
    p, ib = _bufs()
    x = lambda flag: p if flag else None
    return h.lbt_bn_bwd_running(x(g), out, relu, x(k2), 2, 4 * C, C, bits2, ib, x(gq), x(bq), x(run_var), 1e-5, bits_g2,
                                ib if ib_g else None, None, 0, None, bits_g1, ib if ib_g else None, None, 0, None, 0, None, None,
                                x(sums), x(dx), q_grad, gm, gm_lo, 1, kind, None)


def test_bwd_running_rejects_bad_arguments_without_gpu():
    p, ib = _bufs()
    assert _bwd(g=False) == -1                    # no incoming gradient
    assert _bwd(k2=False) == -1                   # no saved k2
    assert _bwd(gq=False) == -1 and _bwd(bq=False) == -1
    assert _bwd(run_var=False) == -1              # no running variance
    assert _bwd(sums=False) == -1                 # no dgamma / dbeta sums
    assert _bwd(ib_g=False) == -1                 # no gradient ranges
    assert _bwd(C=6) == -1 and _bwd(C=0) == -1    # C % 4 != 0
    assert _bwd(relu=2) == -1                     # mask from `out` without `out`
    assert _bwd(relu=3) == -1
    assert _bwd(dx=False) == -1                   # neither fp32 dx nor a gradient quantiser
    assert _bwd(kind=2) == -1                     # neither s8 nor s16 gradients
    assert _bwd(bits2=9) == -1 and _bwd(bits2=1) == -1
    assert _bwd(bits_g2=9) == -1 and _bwd(bits_g1=16) == -1      # wider than 8 bits needs the wide instantiation
    assert _bwd(bits_g2=17, kind=S16) == -1 and _bwd(bits_g1=1, kind=S16) == -1
    q = _lib.QSiteStruct(bits=8, ib=ib.value)
    assert _bwd(dx=False, q_grad=ctypes.addressof(q), gm=None) == -1     # a gradient quantiser without its mantissa buffer
    q16 = _lib.QSiteStruct(bits=16, ib=ib.value)
    assert _bwd(dx=False, q_grad=ctypes.addressof(q16), gm=p) == -1      # 16 bits in the 8-bit instantiation
    assert _bwd(dx=False, q_grad=ctypes.addressof(q16), gm=p, kind=S16) == -1   # 16 bits without the low byte plane
