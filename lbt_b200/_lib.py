"""ctypes binding of liblbt_b200.so (the C ABI declared in include/lbt.h).

There is NO fallback: if the shared library is missing or a call fails, this raises.  PyTorch is
used only for device memory and streams; tensors cross the ABI as raw pointers + sizes.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('LBT_LIB') or os.path.join(_HERE, 'liblbt_b200.so')       # LBT_LIB: an experimental build of the same ABI

c_void_p, c_int, c_size_t, c_float = ctypes.c_void_p, ctypes.c_int, ctypes.c_size_t, ctypes.c_float
c_u64, c_char_p = ctypes.c_uint64, ctypes.c_char_p

# name -> (restype, argtypes); mirrors include/lbt.h one to one (tests/test_abi.py checks both ways)
SIGNATURES = {
    'lbt_version': (c_int, []),
    'lbt_strerror': (c_char_p, [c_int]),
    'lbt_last_cuda_error': (c_char_p, []),
    'lbt_launch_count': (c_u64, []),
    'lbt_quantize': (c_int, [c_void_p, c_size_t, c_size_t, c_int, c_void_p, c_float, c_int, c_void_p, c_u64, c_u64,
                             c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p]),
    'lbt_noise_fill': (c_int, [c_void_p, c_size_t, c_u64, c_u64, c_void_p, c_void_p]),
    'lbt_update_ranges': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    'lbt_step_advance': (c_int, [c_void_p, c_void_p]),
    'lbt_gemm_i8': (c_int, [c_void_p, c_int, c_size_t, c_void_p, c_int, c_size_t, c_size_t, c_size_t, c_size_t, c_int,
                            c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int,
                            c_void_p, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p]),
    'lbt_gemm_i8_dual': (c_int, [c_void_p, c_void_p, c_size_t, c_void_p, c_int, c_size_t, c_size_t, c_size_t, c_size_t, c_void_p,
                                 c_void_p, c_int, c_void_p, c_size_t, c_void_p, c_void_p]),
    'lbt_acc64_finalize': (c_int, [c_void_p, c_size_t, c_void_p, c_void_p, c_int, c_void_p, c_float, c_void_p,
                                   c_void_p]),
    'lbt_im2col_i8': (c_int, [c_void_p, c_int] + [c_int] * 13 + [c_void_p, c_size_t, c_void_p]),
    'lbt_conv_i8_fprop': (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_size_t] + [c_int] * 9 +
                          [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p, c_void_p,
                           c_void_p]),
    'lbt_conv_i8_fprop_dual': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_size_t] + [c_int] * 7 +
                               [c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_void_p, c_void_p]),
    'lbt_conv_i8_dgrad': (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_size_t] + [c_int] * 9 +
                          [c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_void_p, c_void_p]),
    'lbt_conv_i8_wgrad': (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int] + [c_int] * 9 +
                          [c_void_p, c_int, c_int, c_void_p]),
    'lbt_conv_i8_wgrad_dual': (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p] + [c_int] * 9 +
                               [c_void_p, c_int, c_int, c_void_p]),
    'lbt_stem_pack8_bytes': (c_size_t, [c_int, c_int, c_int]),
    'lbt_stem_pack8': (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    'lbt_conv_i8_wgrad_c3': (c_int, [c_void_p, c_int, c_int, c_int, c_void_p] + [c_int] * 8 + [c_void_p, c_int, c_void_p, c_int, c_void_p]),
    'lbt_split_s16': (c_int, [c_void_p, c_size_t, c_void_p, c_void_p, c_void_p]),
    'lbt_transpose_i8': (c_int, [c_void_p, c_size_t, c_size_t, c_size_t, c_void_p, c_size_t, c_void_p]),
    'lbt_colsum_i': (c_int, [c_void_p, c_int, c_size_t, c_size_t, c_void_p, c_void_p]),
    'lbt_bn_bwd_fused': (c_int, [c_void_p, c_void_p]),
    'lbt_maxpool_fwd': (c_int, [c_void_p] + [c_int] * 10 + [c_void_p, c_void_p, c_void_p]),
    'lbt_maxpool_bwd': (c_int, [c_void_p, c_void_p] + [c_int] * 10 + [c_void_p, c_void_p]),
    'lbt_avgpool_fwd': (c_int, [c_void_p] + [c_int] * 8 + [c_void_p, c_void_p]),
    'lbt_avgpool_bwd': (c_int, [c_void_p] + [c_int] * 8 + [c_void_p, c_void_p]),
    'lbt_softmax_xent_fwd': (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    'lbt_softmax_xent_bwd': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    'lbt_relu': (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    'lbt_dropout': (c_int, [c_void_p, c_void_p, c_float, c_u64, c_u64, c_void_p, c_void_p, c_size_t, c_void_p]),
    'lbt_sgd_momentum': (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_float, c_void_p, c_float, c_float,
                                 c_void_p]),
    'lbt_finalize_multi': (c_int, [c_void_p, c_size_t, c_u64, c_void_p]),
    'lbt_noise_fill_multi': (c_int, [c_void_p, c_size_t, c_u64, c_u64, c_void_p, c_void_p]),
    'lbt_param_prep': (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, ctypes.c_uint32, c_u64, c_void_p, c_void_p]),
    'lbt_bn_fwd_quant_stats': (c_int, [c_void_p, c_size_t, c_size_t, c_int, c_int, c_void_p, c_void_p, c_u64, c_u64,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    'lbt_bn_fwd_apply': (c_int, [c_void_p, c_size_t, c_size_t, c_int, c_int, c_void_p, c_void_p, c_float, c_int,
                                 c_void_p, c_void_p, c_u64, c_u64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                 c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, ctypes.c_double, c_int,
                                 c_void_p, c_void_p, c_int, c_void_p]),
    'lbt_bn_fwd_apply2': (c_int, [c_void_p, c_size_t, c_size_t, c_int, c_int, c_void_p, c_void_p, c_float, c_int,
                                  c_void_p, c_void_p, c_u64, c_u64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, ctypes.c_double, c_int,
                                  c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p]),
    # k1, n_outer, H, W, C, bits1, ib1, sums, eps, bits2, ib2, noise2, seed, offset2, dev_step, counters2, gamma_q, beta_q, relu,
    # k2, run_mean, run_var, momentum, stats_minmax, k, s, pad_top, pad_left, POH, POW, pooled, pidx, q_next, next_mant, next_kind, stream
    'lbt_bn_fwd_apply_pooled': (c_int, [c_void_p, c_size_t, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_float, c_int,
                                        c_void_p, c_void_p, c_u64, c_u64, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                        c_void_p, c_void_p, c_void_p, ctypes.c_double, c_int, c_int, c_int, c_int, c_int,
                                        c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    # k1, n_outer, n_inner, C, bits1, ib1, run_mean, run_var, eps, bits2, ib2, noise2, seed, offset2, dev_step, counters2, gamma_q,
    # beta_q, add, relu, k2, out, stats_minmax, q_next, next_mant, next_kind, q_next2, next_mant2, next_kind2, stream
    'lbt_bn_fwd_apply_running': (c_int, [c_void_p, c_size_t, c_size_t, c_int, c_int, c_void_p, c_void_p, c_void_p, c_float, c_int,
                                         c_void_p, c_void_p, c_u64, c_u64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                         c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p]),
    # k1, n_outer, H, W, C, bits1, ib1, run_mean, run_var, eps, bits2, ib2, noise2, seed, offset2, dev_step, counters2, gamma_q,
    # beta_q, relu, k2, stats_minmax, k, s, pad_top, pad_left, POH, POW, pooled, pidx, q_next, next_mant, next_kind, stream
    'lbt_bn_fwd_apply_running_pooled': (c_int, [c_void_p, c_size_t, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                                c_float, c_int, c_void_p, c_void_p, c_u64, c_u64, c_void_p, c_void_p, c_void_p,
                                                c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                                c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    'lbt_bn_bwd_quant_stats': (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_size_t, c_size_t, c_int, c_int,
                                       c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_u64, c_void_p, c_int,
                                       c_void_p, c_void_p, c_u64, c_void_p, c_u64, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_int, c_int, c_void_p]),
    'lbt_bn_bwd_quant_stats_pooled': (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_size_t, c_size_t, c_int, c_int,
                                              c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_u64, c_void_p, c_int,
                                              c_void_p, c_void_p, c_u64, c_void_p, c_u64, c_void_p, c_void_p,
                                              c_void_p, c_int, c_int, c_void_p]),
    'lbt_bn_bwd_apply': (c_int, [c_void_p, c_void_p, c_size_t, c_size_t, c_int, c_int, c_void_p, c_void_p, c_float,
                                 c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    'lbt_conv_i8_dgrad_strided_dual': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_size_t] + [c_int] * 9 +
                                       [c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_void_p, c_void_p]),
    'lbt_conv_i8_dgrad_strided': (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_size_t, c_int, c_int, c_int,
                                          c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_size_t,
                                          c_void_p, c_void_p]),
    'lbt_conv_i8_dgrad_block': (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_size_t] + [c_int] * 9 +
                                [c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_size_t,
                                 c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_void_p, c_void_p]),
    'lbt_dp_step': (c_int, [c_void_p, c_void_p, c_size_t, c_float, c_void_p, c_float, c_int, c_void_p, c_void_p, c_void_p,
                            c_size_t, c_void_p, c_void_p]),
    'lbt_dp_export': (c_int, [c_void_p, c_void_p, c_void_p]),
    'lbt_dp_open': (c_int, [c_void_p, c_void_p]),
    'lbt_dp_close': (c_int, [c_void_p]),
    'lbt_conv_i8_dgrad_bn': (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_size_t] + [c_int] * 7 +
                             [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    'lbt_quantize_residual': (c_int, [c_void_p, c_size_t, c_void_p, c_size_t, c_size_t, c_int, c_void_p, c_int, c_void_p, c_u64,
                                      c_u64, c_void_p, c_void_p, c_void_p, c_void_p]),
    'lbt_augment_batch': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_u64, c_u64,
                                  c_void_p, c_void_p, c_void_p, c_void_p]),
}

# not part of the public header: tuning knobs used by bench sweeps
_INTERNAL = {
    'lbt_quantize_tune': (c_int, [c_int, c_int]),
    'lbt_gemm_debug_error': (c_int, []),
    'lbt_conv_debug_error': (c_int, []),
    'lbt_conv_ldg_debug_error': (c_int, []),
    'lbt_conv_set_path': (c_int, [c_int]),
    'lbt_conv_set_halo': (c_int, [c_int]),
    'lbt_conv_halo_launches': (ctypes.c_longlong, []),
    'lbt_gemm_set_pair': (c_int, [c_int]),
    'lbt_set_pdl': (c_int, [c_int]),
    'lbt_set_carveout': (c_int, [c_int]),
    'lbt_test_fdiv': (c_int, [c_u64, c_u64, c_void_p, c_void_p, c_void_p]),
    'lbt_bn_set_debug': (c_int, [c_void_p]),
    'lbt_conv_ldg_set_debug': (c_int, [c_void_p]),
    'lbt_dp_tune': (c_int, [c_int]),
    'lbt_dp_emulate_scratch_bytes': (c_size_t, [c_int]),
    'lbt_dp_step_emulate': (c_int, [c_int, c_void_p, c_void_p, c_size_t, c_float, c_void_p, c_float, c_int, c_void_p, c_void_p,
                                    c_void_p, c_size_t, c_void_p, c_void_p, c_void_p]),
    'lbt_bn_debug_error': (c_int, []),
}


class LbtError(RuntimeError):
    pass


class FinalizeJob(ctypes.Structure):
    """lbt_finalize_job (include/lbt.h)."""
    _fields_ = [('acc64', c_void_p), ('n', c_u64), ('ibA', c_void_p), ('ibB', c_void_p), ('exp_const', ctypes.c_int32),
                ('add_scale', c_float), ('add', c_void_p), ('out', c_void_p), ('start', c_u64)]


class QSiteStruct(ctypes.Structure):
    """lbt_qsite (include/lbt.h): one quantiser call site as the fused kernels see it."""
    _fields_ = [('bits', ctypes.c_int32), ('stats_minmax', ctypes.c_int32), ('ib', c_void_p), ('noise', c_void_p),
                ('seed', c_u64), ('offset', c_u64), ('dev_step', c_void_p), ('counters', c_void_p)]


class PoolGeom(ctypes.Structure):
    """lbt_pool_geom (include/lbt.h): a max-pool whose backward runs inside lbt_bn_bwd_quant_stats_pooled."""
    _fields_ = [('idx', c_void_p), ('H', ctypes.c_int32), ('W', ctypes.c_int32), ('k', ctypes.c_int32), ('s', ctypes.c_int32),
                ('pad_top', ctypes.c_int32), ('pad_left', ctypes.c_int32), ('OH', ctypes.c_int32), ('OW', ctypes.c_int32)]


class BnBwdLink(ctypes.Structure):
    """lbt_bn_bwd_link (include/lbt.h)."""
    _fields_ = [('q_g2', QSiteStruct), ('q_g1', QSiteStruct), ('bits2', ctypes.c_int32), ('relu', ctypes.c_int32), ('ib2', c_void_p),
                ('gamma_q', c_void_p), ('beta_q', c_void_p), ('k2', c_void_p), ('k1', c_void_p), ('kg1', c_void_p), ('sums', c_void_p)]


class BnBwdArgs(ctypes.Structure):
    """lbt_bn_bwd_args (include/lbt.h)."""
    _fields_ = [('g', c_void_p), ('out', c_void_p), ('k2', c_void_p), ('k1', c_void_p), ('n_outer', c_u64), ('n_inner', c_u64),
                ('C', ctypes.c_int32), ('relu', ctypes.c_int32), ('bits2', ctypes.c_int32), ('bits1', ctypes.c_int32),
                ('ib2', c_void_p), ('ib1', c_void_p), ('gamma_q', c_void_p), ('beta_q', c_void_p), ('q_g2', QSiteStruct),
                ('q_g1', QSiteStruct), ('d_add', c_void_p), ('bwd_sums', c_void_p), ('fwd_sums', c_void_p), ('eps', c_float),
                ('has_q_grad', ctypes.c_int32), ('q_grad', QSiteStruct), ('dx', c_void_p), ('g_mant', c_void_p),
                ('barrier', c_void_p)]


DP_MAX_WORLD, DP_PAD_WORDS, DP_PAD_ERROR, DP_HANDLE_BYTES = 8, 32, 18, 64


class DpPeers(ctypes.Structure):
    """lbt_dp_peers (include/lbt.h)."""
    _fields_ = [('world', ctypes.c_int32), ('rank', ctypes.c_int32), ('grad', c_void_p * DP_MAX_WORLD),
                ('w', c_void_p * DP_MAX_WORLD), ('counters', c_void_p * DP_MAX_WORLD), ('pad', c_void_p * DP_MAX_WORLD)]


class NoiseJob(ctypes.Structure):
    """lbt_noise_job (include/lbt.h)."""
    _fields_ = [('u', c_void_p), ('n', c_u64), ('offset', c_u64), ('start', c_u64)]


class PrepJob(ctypes.Structure):
    """lbt_prep_job (include/lbt.h)."""
    _fields_ = [('x', c_void_p), ('n_outer', c_u64), ('n_inner', c_u64), ('ib', c_void_p), ('counters', c_void_p),
                ('offset', c_u64), ('out_f32', c_void_p), ('out_a', c_void_p), ('out_b', c_void_p), ('ld_a', c_u64),
                ('ld_b', c_u64), ('bits', ctypes.c_int32), ('layout', ctypes.c_int32), ('kh', ctypes.c_uint32),
                ('kw', ctypes.c_uint32), ('Cin', ctypes.c_uint32), ('Cout', ctypes.c_uint32), ('c3pad', ctypes.c_int32),
                ('rot180', ctypes.c_int32), ('sh', ctypes.c_int32), ('sw', ctypes.c_int32)]


def to_device_table(structs, device, keep=None):
    """Upload a list of ctypes Structures as one contiguous device byte tensor.  The staging copy is pinned and
    the transfer asynchronous, so this is legal inside CUDA-graph capture (it becomes a memcpy node; `keep` — a
    list — receives the pinned tensor, which must outlive the graph)."""
    arr = (type(structs[0]) * len(structs))(*structs)
    host = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).pin_memory()
    if keep is not None:
        keep.append(host)
    return host.to(device, non_blocking=True)


_lib = None


def lib():
    """Load (once) and return the ctypes handle.  Raises LbtError if the .so is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LbtError('%s not found — build it with `python -m lbt_b200.build` (needs nvcc); '
                           'there is no CPU or PyTorch fallback for the DFXP hot path' % LIB_PATH)
        h = ctypes.CDLL(LIB_PATH)
        for table in (SIGNATURES, _INTERNAL):
            for name, (res, args) in table.items():
                fn = getattr(h, name)
                fn.restype, fn.argtypes = res, args
        _lib = h
    return _lib


def check(status):
    if status != 0:
        h = lib()
        msg = h.lbt_strerror(status).decode()
        if status == -4:
            msg += ': ' + h.lbt_last_cuda_error().decode()
        raise LbtError('liblbt_b200: %s (status %d)' % (msg, status))


class Profiler:
    """Brackets every C-ABI launch with CUDA events on the launching stream (bench.py's live roofline
    measurement).  ``meta`` carries the algorithmic bytes / ops of the launch."""

    def __init__(self, external=False):
        self.records = []          # (name, start_event, end_event, meta)
        self.keep = []
        self.external = external   # True: events are recorded as nodes of a CUDA graph being captured; every replay
                                   # re-times every launch back to back on the device (no host launch gaps)

    def event(self):
        return torch.cuda.Event(enable_timing=True, external=True) if self.external else torch.cuda.Event(enable_timing=True)

    def summary(self):
        """{name: dict(launches, ms, bytes, ops)} after a synchronize."""
        torch.cuda.synchronize()
        out = {}
        for name, a, b, meta in self.records:
            d = out.setdefault(name, dict(launches=0, ms=0.0, bytes=0, ops=0))
            d['launches'] += 1
            d['ms'] += a.elapsed_time(b)
            d['bytes'] += (meta or {}).get('bytes', 0)
            d['ops'] += (meta or {}).get('ops', 0)
        return out


profiler = None     # set to a Profiler instance to time each launch (never during CUDA-graph capture)


def call(name, *args, meta=None):
    """Invoke one C-ABI entry point and raise on a non-zero status."""
    fn = getattr(lib(), name)
    if profiler is None:
        check(fn(*args))
        return
    a, b = profiler.event(), profiler.event()
    a.record()
    rc = fn(*args)
    b.record()
    profiler.records.append((name, a, b, meta))
    check(rc)


def try_call(name, *args, meta=None):
    """Like call(), but returns False (without raising) when the entry point answers LBT_EUNSUPPORTED — for kernels
    that only take some shapes and have a general path behind them (still inside the library, never a CPU fallback)."""
    fn = getattr(lib(), name)
    if profiler is None:
        rc = fn(*args)
    else:
        a, b = profiler.event(), profiler.event()
        a.record()
        rc = fn(*args)
        b.record()
        if rc == 0:
            profiler.records.append((name, a, b, meta))
        else:
            profiler.keep.append((a, b))     # event nodes already captured into a graph must outlive the capture
    if rc == -2:
        return False
    check(rc)
    return True


def ptr(t):
    """Raw device pointer of a CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise LbtError('lbt_b200 operates on CUDA tensors only (no CPU fallback); got a %s tensor' % t.device)
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def launch_count():
    return int(lib().lbt_launch_count())
