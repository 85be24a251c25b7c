"""CPU-side checks of the eval-mode batch-norm entry points (running statistics): bad arguments are rejected before any
CUDA call, so these run without a GPU."""
import ctypes

from lbt_b200 import _lib


def _bufs():
    f = (ctypes.c_float * 64)()
    p = ctypes.cast(f, ctypes.c_void_p)
    ib = ctypes.cast((ctypes.c_int32 * 1)(2), ctypes.c_void_p)
    return p, ib


def _apply(h, k1, C, run_mean, run_var, gq, out, q_next=None, nm=None, q_next2=None, nm2=None):
    p, ib = _bufs()
    return h.lbt_bn_fwd_apply_running(k1, 2, 4 * C, C, 8, ib, run_mean, run_var, 1e-5, 8, ib, None, 0, 0, None, None, gq, p, None,
                                      1, None, out, 1, q_next, nm, 1 if q_next else 0, q_next2, nm2,
                                      1 if q_next2 else 0, None)


def test_running_apply_rejects_bad_arguments_without_gpu():
    h = _lib.lib()
    p, ib = _bufs()
    assert _apply(h, p, 8, None, p, p, p) == -1           # no running mean
    assert _apply(h, p, 8, p, None, p, p) == -1           # no running variance
    assert _apply(h, None, 8, p, p, p, p) == -1           # no k1
    assert _apply(h, p, 8, p, p, None, p) == -1           # no gamma
    assert _apply(h, p, 6, p, p, p, p) == -1              # C % 4 != 0
    assert _apply(h, p, 0, p, p, p, p) == -1
    assert _apply(h, p, 8, p, p, p, None) == -1           # neither an fp32 output nor a consumer quantiser
    q2 = _lib.QSiteStruct(bits=9, ib=ib.value)
    assert _apply(h, p, 8, p, p, p, p, q_next2=ctypes.addressof(q2), nm2=p) == -1   # second consumer without a first


def test_running_pooled_rejects_bad_arguments_without_gpu():
    h = _lib.lib()
    p, ib = _bufs()

    def pooled(run_mean, run_var, C=64, k1=p, pidx=p):
        return h.lbt_bn_fwd_apply_running_pooled(k1, 2, 16, 16, C, 8, ib, run_mean, run_var, 1e-5, 8, ib, None, 0, 0, None, None,
                                                 p, p, 1, None, 1, 3, 2, 0, 0, 8, 8, p, pidx, None, None, 0, None)

    assert pooled(None, p) == -1
    assert pooled(p, None) == -1
    assert pooled(p, p, k1=None) == -1
    assert pooled(p, p, pidx=None) == -1
    assert pooled(p, p, C=62) == -1                        # C % 4 != 0
    assert pooled(p, p, C=32) == -2                        # outside the stem's shape class: LBT_EUNSUPPORTED, as for training
