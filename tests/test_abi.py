"""CPU-side checks of the drop-in boundary: the .so loads and exports exactly what include/lbt.h declares."""
import ctypes
import os
import re

from lbt_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, 'include', 'lbt.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return set(re.findall(r'\b(lbt_[a-z0-9_]+)\s*\(', src))


def test_library_builds_and_loads():
    from lbt_b200 import build
    path = build.build()
    assert os.path.exists(path)
    h = _lib.lib()
    assert h.lbt_version() == 100
    assert h.lbt_strerror(0) == b'ok'
    assert b'invalid' in h.lbt_strerror(-1)


def test_every_declared_symbol_is_exported_and_bound():
    h = ctypes.CDLL(_lib.LIB_PATH)
    declared = _declared()
    assert declared, 'no declarations parsed from include/lbt.h'
    for name in declared:
        assert hasattr(h, name), 'include/lbt.h declares %s but liblbt_b200.so does not export it' % name
    assert declared == set(_lib.SIGNATURES), (declared ^ set(_lib.SIGNATURES))


def test_argument_validation_without_gpu():
    h = _lib.lib()
    # null tensor / bad bits are rejected before any CUDA call
    assert h.lbt_quantize(None, 1, 1, 8, None, 0.0, 0, None, 0, 0, None, None, None, 0, None, 0, None) == -1
    buf = (ctypes.c_float * 4)()
    ib = (ctypes.c_int32 * 1)(2)
    p = ctypes.cast(buf, ctypes.c_void_p)
    q = ctypes.cast(ib, ctypes.c_void_p)
    assert h.lbt_quantize(p, 1, 4, 0, q, 0.0, 0, None, 0, 0, None, p, None, 0, None, 0, None) == -1     # bits < 1
    assert h.lbt_quantize(p, 1, 4, 32, q, 0.0, 0, None, 0, 0, None, p, None, 0, None, 0, None) == -1    # bits > 31 (32 = the caller's pass-through)
    assert h.lbt_quantize(p, 1, 4, 8, q, 0.0, 1, None, 0, 0, None, p, None, 0, None, 0, None) == -1     # noise mode, no noise
    assert h.lbt_quantize(p, 1, 4, 9, q, 0.0, 0, None, 0, 0, None, None, p, 1, None, 0, None) == -1     # 9 bits into s8
    assert h.lbt_quantize(p, 1, 4, 8, q, 0.0, 0, None, 0, 0, None, p, None, 0, None, 1, None) == -1     # update w/o counters
    assert h.lbt_quantize(p, 0, 4, 8, q, 0.0, 0, None, 0, 0, None, p, None, 0, None, 0, None) == 0      # empty tensor


def test_cpu_tensor_is_an_error():
    import pytest
    import torch
    from lbt_b200 import quantizer
    with pytest.raises(_lib.LbtError):
        quantizer.quantize(torch.zeros(4, 4), 8, torch.tensor(2, dtype=torch.int32))


def test_dp_augment_and_residual_entry_points_validate_arguments_without_gpu():
    """lbt_dp_step / lbt_augment_batch / lbt_quantize_residual reject bad arguments before any CUDA call."""
    h = _lib.lib()
    buf = (ctypes.c_float * 16)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    ib = ctypes.cast((ctypes.c_int32 * 1)(2), ctypes.c_void_p)
    # data-parallel step: null descriptor, world out of range, rank out of range
    assert h.lbt_dp_step(None, p, 16, 0.1, None, 0.9, 0, None, None, None, 0, None, None) == -1
    peers = _lib.DpPeers()
    peers.world, peers.rank = 9, 0
    assert h.lbt_dp_step(ctypes.addressof(peers), p, 16, 0.1, None, 0.9, 0, None, None, None, 0, None, None) == -1
    peers.world, peers.rank = 2, 2
    assert h.lbt_dp_step(ctypes.addressof(peers), p, 16, 0.1, None, 0.9, 0, None, None, None, 0, None, None) == -1
    assert h.lbt_dp_export(None, None, None) == -1 and h.lbt_dp_open(None, None) == -1 and h.lbt_dp_close(None) == -1
    # input pipeline: null images, negative pad; an empty batch is a no-op
    assert h.lbt_augment_batch(None, None, None, 4, 8, 8, 3, 4, 1, None, 0, 0, None, None, p, None) == -1
    assert h.lbt_augment_batch(p, None, None, 4, 8, 8, 3, -1, 1, None, 0, 0, None, None, p, None) == -1
    assert h.lbt_augment_batch(p, None, None, 0, 8, 8, 3, 4, 1, None, 0, 0, None, None, p, None) == 0
    # error-feedback quantiser: more gradient rows than buffer rows, bad bits, noise mode without noise; empty is a no-op
    assert h.lbt_quantize_residual(p, 3, p, 2, 4, 8, ib, 0, None, 0, 0, None, p, None, None) == -1
    assert h.lbt_quantize_residual(p, 1, p, 2, 4, 0, ib, 0, None, 0, 0, None, p, None, None) == -1
    assert h.lbt_quantize_residual(p, 1, p, 2, 4, 8, ib, 1, None, 0, 0, None, p, None, None) == -1
    assert h.lbt_quantize_residual(p, 0, p, 0, 4, 8, ib, 0, None, 0, 0, None, p, None, None) == 0


def test_dp_struct_mirrors_match_the_header():
    assert ctypes.sizeof(_lib.DpPeers) == 8 + 4 * 8 * 8
    assert _lib.DP_PAD_WORDS * 4 <= 256 and _lib.DP_HANDLE_BYTES == 64
