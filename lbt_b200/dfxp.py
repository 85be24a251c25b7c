"""Quantised layers of the DFXP training path — PyTorch host side over liblbt_b200's C ABI.

Mirrors the reference's layer set (``dfxp:N`` = /root/reference/dynamic_fixed_point.py:N) with the
PyTorch-style constructors the reference's orphan ``custom.py`` expects (custom.py:5, 11-12, 29-30):

    Conv2d_q(bits, in_channels, out_channels, kernel_size, stride=1, padding='SAME', bias=True)   dfxp:224-316
    Linear_q(bits, in_features, out_features, bias=True)           (= Dense_q)                    dfxp:319-470
    BatchNorm2d_q(bits, num_features)    (= Normalization_q + Rescale_q, BatchNorm_q)             dfxp:539-743
    ResidualBlock_q / ResidualBottleneck_q                                                        dfxp:746-980

Semantics follow the TensorFlow classes: NHWC/HWIO arithmetic (tensors are logical NCHW stored
channels_last, conv weights are stored HWIO, dense weights [in, out]) so the rounding noise
broadcasts over dim 0 exactly as ``tf.random_uniform(X.shape[1:])`` does; conv activations use
``bits+1`` (dfxp:287); every quantiser is stochastic (dfxp:192-206 hard-code it); the backward
pass quantises the incoming gradient, is straight-through for the forward quantisers, and carries
the weight decay inside the gradient (``+ 2*wd*W``, dfxp:302).

All arithmetic on tensors runs in the library's kernels (quantiser, im2col, tcgen05 int8 GEMM);
there is no PyTorch/CPU fallback for them.  Range variables stay constant during a step and are
advanced once per step by ``Runtime.update_ranges()`` (read-then-update, SURVEY.md App. E-1).
"""
import contextlib
import ctypes
import os
import math

import torch
import torch.nn as nn

from . import _lib, gemm as G, quantizer as Q


# ------------------------------------------------------------------------------------------------
# Runtime: shared per-model state (quantiser ids, Philox seed, device step counter, flat range state)
# ------------------------------------------------------------------------------------------------


class Runtime:
    """What the TF graph + session held implicitly: the list of quantisers ('update_range'
    collection, dfxp:40-41), the RNG stream and the per-step range update (trainer.py:63, 157)."""

    def __init__(self, seed=0):
        self.seed = int(seed)
        self.sites = []
        self.dev_step = None         # int64[1] on the device once finalised
        self.noise_fn = None         # tests: callable(site, n_inner, device) -> explicit noise tensor
        self.flat = None
        self.grad_sink = None        # Trainer: collects every integer gradient sum for ONE lbt_finalize_multi launch
        self.prep = None             # ParamPrep: ONE lbt_param_prep launch quantises + packs every parameter
        self._arena = None           # int64 workspace (integer sums), zeroed once per step
        self._arena_off = 0
        self._arena_used = 0
        self._arena_on = False
        self._side = None            # side stream: wgrad runs beside dgrad (independent consumers of the same gradient)
        self.overlap = True
        self._prep_pending = False   # begin_step() left the parameter branch running on the side stream
        self._prep_head_pending = False
        self._prep_ev = None
        self._noise_req = {}         # (quantiser id, n_inner) wanted by fused tensor-core epilogues
        self._noise_tab = None       # dict(map={key: fp32 view}, jobs=device table, total=groups, keep=[...])
        self._noise_valid = False
        self._n_dropout = 0          # dropout sites are numbered per runtime, like the quantisers (reproducible across processes)

    def next_dropout_id(self):
        d = self._n_dropout
        self._n_dropout += 1
        return d

    # ---- per-step noise arena: ONE launch fills the noise vectors the conv epilogues read (same Philox stream) ----
    def noise_for(self, site, n_inner, device):
        """The [n_inner] noise vector of `site` for the current step, or None (the kernel then runs Philox itself).
        Only inside a Trainer step; a vector requested for the first time is available from the next step on."""
        if self.noise_fn is not None or not self._arena_on:
            return None
        key = (site.qid, int(n_inner))
        tab = self._noise_tab
        if tab is not None and self._noise_valid and key in tab['map']:
            self.join_prep(head=True)
            return tab['map'][key]
        self._noise_req[key] = True
        return None

    def _fill_noise(self, device):
        if not self._noise_req:
            return
        tab = self._noise_tab
        if tab is None or any(k not in tab['map'] for k in self._noise_req):
            keys = sorted(self._noise_req)
            total = sum(-(-n // 4) for _, n in keys)
            arena = torch.empty(total * 4, dtype=torch.float32, device=device)
            jobs, m, start = [], {}, 0
            for qid, n in keys:
                u = arena[start * 4:start * 4 + n]
                m[(qid, n)] = u
                jobs.append(_lib.NoiseJob(u=u.data_ptr(), n=n, offset=Q.make_offset(qid, 0), start=start))
                start += -(-n // 4)
            keep = []
            tab = dict(map=m, jobs=_lib.to_device_table(jobs, device, keep=keep), njobs=len(jobs), total=total,
                       arena=arena, keep=keep)
            self._noise_tab = tab
        _lib.call('lbt_noise_fill_multi', _lib.ptr(tab['jobs']), tab['njobs'], tab['total'], self.seed,
                  _lib.ptr(self.dev_step), _lib.stream())
        self._noise_valid = True

    # ---- per-step workspace: exact integer sums live in one arena that is zeroed with a single launch ----
    def begin_step(self, device):
        """Start of a training step: recycle + zero the int64 arena, then quantise and pack all parameters."""
        need = max(self._arena_off, 1 << 14)
        if self._arena is None or self._arena.numel() < need or self._arena.device != torch.device(device):
            self._arena = torch.zeros(need * 5 // 4, dtype=torch.int64, device=device)
        elif self._arena_used:
            self._arena[:self._arena_used].zero_()
        self._arena_off = 0
        self._arena_used = 0
        self._arena_on = True
        self._prep_valid = False
        # the parameter side (quantise + pack every weight, fill the noise vectors) shares nothing with the quantisation of
        # the step's input, so inside a Trainer step it runs as a parallel branch; its first consumer joins (join_prep)
        fork = (self.prep is not None and self.overlap and self.grad_sink is not None and _lib.profiler is None
                and os.environ.get('LBT_PREP_FORK', '1') != '0')
        if fork:
            main, side = torch.cuda.current_stream(device), self.side_stream(device)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                self._fill_noise(device)
                self.prep.run('head')
                self._prep_ev = torch.cuda.Event()
                self._prep_ev.record(side)          # noise vectors + the first layer's operands: all the first kernels need
                self.prep.run('rest')
            self._prep_valid = True
            self._prep_pending = True
            self._prep_head_pending = True
            return
        if self.prep is not None:
            self.prep.run()
            self._prep_valid = True      # until update_ranges() closes the step
        self._fill_noise(device)

    def join_prep(self, layer=None, head=False):
        """First consumer of a prepared operand or a noise vector: wait for the parameter branch of begin_step() — for its
        head only (noise vectors and the first layer's operands, an event in the middle of the branch) when that is all the
        consumer needs."""
        if not self._prep_pending:
            return
        main = torch.cuda.current_stream(self._side.device)
        if head or (layer is not None and self.prep is not None and layer in self.prep.head):
            if self._prep_head_pending:
                self._prep_head_pending = False
                main.wait_event(self._prep_ev)
            return
        self._prep_pending = self._prep_head_pending = False
        main.wait_stream(self._side)

    def zeros_i64(self, n, device):
        """n zeroed int64 slots (16-byte aligned) from the arena; a fresh tensor when the arena is off or full."""
        if not self._arena_on:
            return torch.zeros(int(n), dtype=torch.int64, device=device)
        n_al = (int(n) + 1) & ~1
        off = self._arena_off
        self._arena_off += n_al                      # keeps counting so the next begin_step() can grow the arena
        if self._arena_on and off + n_al <= self._arena.numel():
            self._arena_used = off + n_al
            return self._arena[off:off + n]
        return torch.zeros(int(n), dtype=torch.int64, device=device)

    def join_side(self):
        """Make the current stream wait for the weight-gradient kernels still running on the side stream."""
        if getattr(self, '_side_pending', False) and self._side is not None:
            torch.cuda.current_stream(self._side.device).wait_stream(self._side)
        self._side_pending = False

    def side_stream(self, device):
        if self._side is None or self._side.device != torch.device(device):
            self._side = torch.cuda.Stream(device=device)
        return self._side

    def register(self, site):
        site.qid = len(self.sites)
        self.sites.append(site)

    def finalize(self, device, counters=None):
        """Flatten every quantiser's range/counters into contiguous device arrays (one
        lbt_update_ranges launch per step; one exchange of the counters under data parallelism).
        ``counters``: zeroed int64 [n, CNT_WORDS] storage to use (the peer-mapped arena of lbt_b200.dp)."""
        n = len(self.sites)
        ranges = torch.empty(n, dtype=torch.int32, device=device)
        if counters is None:
            counters = torch.zeros(n, Q.CNT_WORDS, dtype=torch.int64, device=device)
        assert counters.shape == (n, Q.CNT_WORDS) and counters.dtype == torch.int64
        bits = torch.tensor([s.bits for s in self.sites], dtype=torch.int32, device=device)
        target = torch.tensor([s.target for s in self.sites], dtype=torch.float32, device=device)
        for i, s in enumerate(self.sites):
            ranges[i] = int(s.range)
            s._buffers['range'] = ranges[i]
            s._buffers['counters'] = counters[i]
        self.flat = dict(ranges=ranges, counters=counters, bits=bits, target=target)
        self.dev_step = torch.zeros(1, dtype=torch.int64, device=device)
        return self

    def update_ranges(self):
        """The ``update_range_op`` fetch of trainer.py:157 for all quantisers, then step += 1."""
        f = self.flat
        _lib.call('lbt_update_ranges', _lib.ptr(f['ranges']), _lib.ptr(f['counters']), _lib.ptr(f['bits']),
                                       _lib.ptr(f['target']), len(self.sites), _lib.stream())
        _lib.call('lbt_step_advance', _lib.ptr(self.dev_step), _lib.stream())
        self.close_step()

    def close_step(self):
        self.join_prep()
        self._arena_on = False           # the step is closed: prepared operands and arena slices are stale now
        self._prep_valid = False
        self._noise_valid = False

    def ranges(self):
        """{quantiser name: integer_bits} — the cheap parity probe (tf.summary of *_range, dfxp:180-190)."""
        vals = self.flat['ranges'].cpu().tolist() if self.flat is not None else [int(s.range) for s in self.sites]
        return {s.name: v for s, v in zip(self.sites, vals)}


class ParamPrep:
    """All parameter quantisers of a step in ONE launch (lbt_param_prep): conv / dense weights are quantised
    (dfxp:289, 386) and written straight into the packed operand layouts the tensor-core kernels read; biases
    and BN gamma / beta (dfxp:294, 391, 679-682) become fake-quant fp32 vectors.  Same quantiser ids, ranges and
    Philox stream as the per-layer path, so the results are identical bit for bit."""

    CHUNK = 4096

    def __init__(self, model, runtime, device):
        self.rt = runtime
        self.entries = {}            # module -> dict of prepared tensors
        self._njobs_of = {}          # module -> number of jobs it contributed (jobs are in module order)
        self.head, self.head_blocks = set(), 0
        jobs = []

        def job(site, x, layout=0, **kw):
            n_outer, n_inner = Q.rows_view(x)
            j = _lib.PrepJob(x=x.data_ptr(), n_outer=n_outer, n_inner=n_inner, ib=site.range.data_ptr(),
                             counters=site.counters.data_ptr(), offset=Q.make_offset(site.qid, 0), bits=site.bits,
                             layout=layout, **kw)
            jobs.append(j)

        def vec(site, p):
            out = torch.empty_like(p.data)
            job(site, p.data, out_f32=out.data_ptr())
            return out

        for m in model.modules():
            n_before = len(jobs)
            if isinstance(m, Conv2d_q) and m.qW.bits <= 8:
                kh, kw, Cin, Cout = m.weight.shape
                e = {}
                c3 = bool(m.input_signed and m.qX.bits == 9 and Cin == 3 and m.implicit and _implicit_ok(Cout, 1, 1))
                Ka = kh * kw * (16 if c3 else Cin)
                e['c3'] = c3
                e['wt'] = torch.zeros(Cout, _pitch16(Ka), dtype=torch.int8, device=device)[:, :Ka]
                rot = bool(m.implicit and m.stride == (1, 1) and _implicit_ok(Cout, kh, kw) and not (kh == 1 and kw == 1))
                cls = _dgrad_classes_ok(m, Cin, Cout, kh, kw, m.stride[0], m.stride[1])
                K2 = kh * kw * Cout
                e['rot180'] = rot
                e['classes'] = cls
                e['w2'] = None if c3 else torch.zeros(Cin, _pitch16(K2), dtype=torch.int8, device=device)[:, :K2]
                job(m.qW, m.weight.data, layout=1, kh=kh, kw=kw, Cin=Cin, Cout=Cout, c3pad=int(c3), rot180=2 if cls else int(rot),
                    sh=m.stride[0], sw=m.stride[1],
                    out_a=e['wt'].data_ptr(), ld_a=e['wt'].stride(0),
                    out_b=0 if e['w2'] is None else e['w2'].data_ptr(), ld_b=0 if e['w2'] is None else e['w2'].stride(0))
                if m.bias is not None:
                    e['bq'] = vec(m.qb, m.bias)
                self.entries[m] = e
            elif isinstance(m, Linear_q) and m.qW.bits <= 8:
                In, Out = m.weight.shape
                e = {}
                e['wt'] = torch.zeros(Out, _pitch16(In), dtype=torch.int8, device=device)[:, :In]
                e['w2'] = torch.zeros(In, _pitch16(Out), dtype=torch.int8, device=device)[:, :Out]
                job(m.qW, m.weight.data, layout=2, Cin=In, Cout=Out, out_a=e['wt'].data_ptr(), ld_a=e['wt'].stride(0),
                    out_b=e['w2'].data_ptr(), ld_b=e['w2'].stride(0))
                if m.bias is not None:
                    e['bq'] = vec(m.qb, m.bias)
                self.entries[m] = e
            elif isinstance(m, Rescale_q):
                self.entries[m] = dict(gq=vec(m.qg, m.gamma), bq=vec(m.qb, m.beta))
            if m in self.entries:
                self._njobs_of[m] = len(jobs) - n_before
        self.njobs = len(jobs)
        if not jobs:
            return
        # head: the first weight layer and the batch-norm behind it — what the first kernels of the forward pass need.  Their
        # jobs come first (module order), so the launch can be cut in two: the step's first convolution waits for the head only
        # while the rest of the parameters is prepared beside it (Runtime.begin_step / join_prep)
        ents = list(self.entries)
        self.head = set(ents[:1])
        if len(ents) > 1 and isinstance(ents[1], Rescale_q):
            self.head.add(ents[1])
        head_jobs = sum(self._njobs_of[m] for m in self.head)
        bj, bc = [], []
        self.head_blocks = 0
        for i, j in enumerate(jobs):
            n = j.n_outer * j.n_inner
            for c in range(-(-n // self.CHUNK)):
                bj.append(i)
                bc.append(c)
            if i + 1 == head_jobs:
                self.head_blocks = len(bj)
        self.jobs_dev = _lib.to_device_table(jobs, device)
        self.block_job = torch.tensor(bj, dtype=torch.int32, device=device)
        self.block_chunk = torch.tensor(bc, dtype=torch.int32, device=device)
        self._keep = jobs

    def run(self, part=None):
        """part: None = everything in one launch; 'head' / 'rest' = the two halves of the cut described above."""
        if not self.njobs:
            return
        rt = self.rt
        nb, hb = self.block_job.numel(), self.head_blocks
        lo, hi = (0, nb) if part is None else ((0, hb) if part == 'head' else (hb, nb))
        if hi <= lo:
            return
        _lib.call('lbt_param_prep', _lib.ptr(self.jobs_dev), self.block_job.data_ptr() + 4 * lo, self.block_chunk.data_ptr() + 4 * lo,
                  hi - lo, self.CHUNK, rt.seed, _lib.ptr(rt.dev_step), _lib.stream())


def _prepared(layer):
    """The ParamPrep entry of a layer for the current step, or None (per-layer quantisers run instead)."""
    rt = layer.qX.runtime
    if rt.prep is None or rt.noise_fn is not None or not getattr(rt, '_prep_valid', False):
        return None
    rt.join_prep(layer)
    return rt.prep.entries.get(layer)


def _emit_grad(rt, param, acc, *, ibA=None, ibB=None, exp_const=0, add_scale=0.0, shape=None):
    """Gradient of ``param`` from its exact integer sum: handed to the Trainer's sink (one lbt_finalize_multi per
    step) when there is one, else finalised here.  ``+ 2*wd*param`` rides along (dfxp:302, 457, 689)."""
    sink = rt.grad_sink
    if sink is not None and sink.accepts(param):
        sink.add(param, acc, ibA, ibB, exp_const, add_scale)
        return None
    g = G.acc64_finalize(acc, ibA=ibA, ibB=ibB, exp_const=exp_const, add=param.detach().reshape(-1) if add_scale else None,
                         add_scale=add_scale)
    return g.view(shape if shape is not None else param.shape)


_default_runtime = Runtime()


def default_runtime():
    return _default_runtime


class QuantSite(nn.Module):
    """One ``weight_quantization`` call site and its ``*_range`` variable (dfxp:161-171)."""

    def __init__(self, runtime, name, bits, init_range=2, target_overflow_rate=0.0):
        super().__init__()
        assert 1 <= bits <= 32, 'invalid value for bits: %d' % bits          # dfxp:21
        self.runtime = runtime
        self.name = name
        self.bits = int(bits)
        self.target = float(target_overflow_rate)
        self.register_buffer('range', torch.tensor(int(init_range), dtype=torch.int32))
        self.register_buffer('counters', torch.zeros(Q.CNT_WORDS, dtype=torch.int64))
        runtime.register(self)

    def quantize(self, x, want_fp32=True, mant_kind=Q.MANT_NONE, out_mant=None):
        """Stochastic DFXP quantisation of ``x`` (memory order = TF layout).  Gathers the overflow
        counters; the range itself moves in Runtime.update_ranges()."""
        rt = self.runtime
        kw = dict(target_overflow_rate=self.target, want_fp32=want_fp32, mant_kind=mant_kind, counters=self.counters,
                  update_range=False, out_mant=out_mant)
        if rt.noise_fn is not None:
            n_inner = Q.rows_view(x)[1]
            kw.update(mode=Q.ROUND_NOISE, noise=rt.noise_fn(self, n_inner, x.device))
        else:
            kw.update(mode=Q.ROUND_PHILOX, seed=rt.seed, offset=Q.make_offset(self.qid, 0), dev_step=rt.dev_step)
        if self.target == 0.0:      # the controller then only tests "any overflow": min/max statistics suffice
            kw['mode'] |= Q.STATS_MINMAX
        return Q.quantize(x, self.bits, self.range, **kw)

    def abi(self, n_inner, device, arena=False):
        """This call site as an ``lbt_qsite`` for the fused kernels (same ids, ranges, Philox stream and
        statistics block as quantize(), so fused and unfused runs are bit-identical).  arena=True: take the
        step's pre-generated noise vector when the runtime has one (tensor-core epilogues)."""
        rt = self.runtime
        qs = _lib.QSiteStruct(bits=self.bits, stats_minmax=int(self.target == 0.0), ib=self.range.data_ptr(),
                              noise=0, seed=rt.seed, offset=Q.make_offset(self.qid, 0),
                              dev_step=_lib.ptr(rt.dev_step) or 0, counters=self.counters.data_ptr())
        if rt.noise_fn is not None:
            nz = rt.noise_fn(self, n_inner, device).contiguous()
            qs.noise, qs.offset = nz.data_ptr(), 0
            qs._keep = nz                 # the kernel is stream-ordered before the allocator can reuse it
        elif arena:
            nz = rt.noise_for(self, n_inner, device)
            if nz is not None:
                qs.noise = nz.data_ptr()
        return qs

    def extra_repr(self):
        return '%s bits=%d' % (self.name, self.bits)


class _QuantSTE(torch.autograd.Function):
    """Forward: fake-quantise through the site.  Backward: identity (dfxp:30, 38)."""

    @staticmethod
    def forward(ctx, x, site):
        q, _ = site.quantize(x)
        return q

    @staticmethod
    def backward(ctx, dy):
        return dy, None


class _GradQuant(torch.autograd.Function):
    """Identity in forward; quantises the incoming gradient in backward (``gradq``, dfxp:300, 621, 687)."""

    @staticmethod
    def forward(ctx, y, site):
        ctx.site = site
        return y.view_as(y)

    @staticmethod
    def backward(ctx, dy):
        dy = _mem_contig(dy)
        q, _ = ctx.site.quantize(dy)
        return q, None


def _require_cuda_f32(x, who):
    """The path has no CPU / PyTorch fallback (SURVEY §8b): anything but an fp32 CUDA tensor is an error."""
    if not x.is_cuda or x.dtype != torch.float32:
        raise _lib.LbtError('%s: expects an fp32 CUDA tensor (got %s on %s); there is no CPU or PyTorch fallback'
                            % (who, x.dtype, x.device))


def _mem_contig(x):
    """Contiguous in memory in the TF order: channels_last for 4-D (NHWC), plain otherwise."""
    if x.dim() == 4:
        return x if x.is_contiguous(memory_format=torch.channels_last) else x.contiguous(memory_format=torch.channels_last)
    return x.contiguous()


def same_pad(in_size, k, s):
    """TF 'SAME': (out, pad_before, pad_after) — pad_total = max((out-1)*s + k - in, 0), before = total//2."""
    out = -(-in_size // s)
    total = max((out - 1) * s + k - in_size, 0)
    return out, total // 2, total - total // 2


def _pitch16(k):
    return -(-k // 16) * 16


def _as_operand(t):
    """[rows, K] byte matrix with a 16-byte row pitch (TMA requirement); copies only when needed."""
    rows, K = t.shape
    if t.stride(1) == 1 and t.stride(0) % 16 == 0 and t.data_ptr() % 16 == 0:
        return t
    buf = torch.zeros(rows, _pitch16(K), dtype=t.dtype, device=t.device)
    buf[:, :K] = t
    return buf[:, :K]


def _transpose_bytes(t):
    """[R, C] -> [C, R] byte matrix with a 16-byte pitch (lbt_transpose_i8)."""
    R, C = t.shape
    assert t.stride(1) == 1
    out = torch.empty(C, _pitch16(R), dtype=t.dtype, device=t.device)
    _lib.call('lbt_transpose_i8', _lib.ptr(t), R, C, t.stride(0), _lib.ptr(out), out.stride(0), _lib.stream())
    return out[:, :R]


def _im2col(src_nhwc, src_kind, OH, OW, kh, kw, sh, sw, pt, pl, transposed):
    N, H, W, C = src_nhwc.shape
    segs = 3 if src_kind == Q.MANT_S16 else 1
    K = kh * kw * C * segs
    M = N * OH * OW
    out = torch.empty(M, _pitch16(K), dtype=torch.int8 if src_kind != Q.MANT_U8 else torch.uint8, device=src_nhwc.device)
    _lib.call('lbt_im2col_i8', _lib.ptr(src_nhwc), src_kind, N, H, W, C, OH, OW, kh, kw, sh, sw, pt, pl,
                                        1 if transposed else 0, _lib.ptr(out), out.stride(0), _lib.stream())
    return out[:, :K]


def _colsum(mant2d, kind, rt=None):
    acc = (rt.zeros_i64(mant2d.shape[1], mant2d.device) if rt is not None
           else torch.zeros(mant2d.shape[1], dtype=torch.int64, device=mant2d.device))
    _lib.call('lbt_colsum_i', _lib.ptr(mant2d), kind, mant2d.shape[0], mant2d.shape[1], _lib.ptr(acc),
                                       _lib.stream())
    return acc


def _implicit_ok(C, kh, kw):
    """Shapes the implicit-GEMM kernel takes: C in {16,32,64} or a multiple of 128; kh*kw*C <= 65536."""
    return (C in (16, 32, 64) or (C >= 128 and C % 128 == 0)) and kh * kw * C <= 65536 and kh <= 255 and kw <= 255


def _gather_ok(C, Cout, kh, kw):
    """Shapes of the cp.async-gather kernel (csrc/conv_ldg.cu): gathered channels 16/32/64, <= 128 output channels,
    filter bank resident in shared memory."""
    if C not in (16, 32, 64) or not 1 <= Cout <= 128:
        return False
    kcp = (kh * kw * (C // 16) + 1) & ~1
    bn = 16 if Cout <= 16 else (32 if Cout <= 32 else (64 if Cout <= 64 else 128))
    return kcp * bn * 16 + 2 * 16384 + 1024 <= 200 * 1024 and kh * kw * C <= 65536 and kcp <= 256 and kh * kw <= 64 and kh <= 16 and kw <= 16


def _class_perm(kh, kw, sh, sw):
    """Filter taps in the parity-class order of csrc/conv_classes.h (the operand of lbt_conv_i8_dgrad_strided)."""
    perm = []
    for r0 in range(sh):
        for s0 in range(sw):
            for r in reversed(range(r0, kh, sh)):
                for s_ in reversed(range(s0, kw, sw)):
                    perm.append(r * kw + s_)
    return perm


DGRAD_CLASSES = True      # module switch (tests): strided input gradients with wide gathered channels as parity-class sub-convolutions


def _dgrad_classes_ok(layer, Cin, Cout, kh, kw, sh, sw):
    """Strided input gradients that run as stride-1 sub-convolutions per parity class (lbt_conv_i8_dgrad_strided) instead of
    a transposed im2col matrix + GEMM: everything the gather kernel does not take."""
    if layer.qG.bits > 8:      # 16-bit gradients: the classes run on the dual-accumulator kernels (lbt_conv_i8_dgrad_strided_dual)
        return (DGRAD_CLASSES and DUAL_HALO and layer.implicit and (sh, sw) != (1, 1) and sh <= 4 and sw <= 4 and layer.qG.bits <= 16 and
                layer.qW.bits <= 8 and (Cout == 64 or Cout % 128 == 0) and Cin >= 64 and Cin % 4 == 0)
    return (DGRAD_CLASSES and layer.implicit and (sh, sw) != (1, 1) and sh <= 4 and sw <= 4 and layer.qG.bits <= 8 and
            layer.qW.bits <= 8 and (Cout in (16, 32, 64) or Cout % 128 == 0) and Cin % 4 == 0 and
            not _gather_ok(Cout, Cin, kh, kw))


# conv -> BN -> ReLU -> 3x3/2 max-pool: BN pass 2 and the pool in one kernel (LBT_FUSE_POOL_FWD=0: two launches and an fp32 tensor).
FUSE_POOL_FWD = os.environ.get('LBT_FUSE_POOL_FWD', '1') != '0'

# First-layer weight gradient through lbt_conv_i8_wgrad_c3 (LBT_STEM_WGRAD=0: the general kernel on the 16-byte pixels).
STEM_WGRAD = os.environ.get('LBT_STEM_WGRAD', '1') != '0'

def _conv_implicit(src_nhwc, src_kind, wp, Cout, kh, kw, sh, sw, pt, pl, OH, OW, ib_src, ib_w, exp_const, bias, out2d,
                   bnq=None, addend=None):
    """lbt_conv_i8_fprop: out2d[N*OH*OW, Cout] = conv(src, wp) * 2^(exp_const + ib_src + ib_w) (+ bias), or with
    ``bnq = (QSiteStruct, k_out, sums)`` the fused re-quantising epilogue (s8 mantissas + batch statistics)."""
    N, H, W, C = src_nhwc.shape
    qs, k_out, sums = bnq if bnq is not None else (None, None, None)
    _lib.call('lbt_conv_i8_fprop', _lib.ptr(src_nhwc), src_kind, N, H, W, C, _lib.ptr(wp), Q.MANT_S8, wp.stride(0), Cout,
              kh, kw, sh, sw, pt, pl, OH, OW, _lib.ptr(ib_src), _lib.ptr(ib_w), int(exp_const), _lib.ptr(bias),
              _lib.ptr(out2d), out2d.stride(0) if out2d is not None else Cout,
              ctypes.addressof(qs) if qs is not None else None, _lib.ptr(k_out), _lib.ptr(sums), _lib.ptr(addend), _lib.stream(),
              meta=dict(ops=2 * N * OH * OW * Cout * kh * kw * C,
                        bytes=N * H * W * C + Cout * kh * kw * C + N * OH * OW * Cout * (1 if qs is not None else 4)))


# ------------------------------------------------------------------------------------------------
# Conv2d_q
# ------------------------------------------------------------------------------------------------


def _conv_geom(layer, x, weight):
    """(N, H, W, Cin, Cout, kh, kw, sh, sw, pad_top, pad_left, OH, OW) of a Conv2d_q call on logical-NCHW ``x``."""
    N, Cin, H, W = x.shape
    kh, kw, _, Cout = weight.shape
    sh, sw = layer.stride
    if layer.padding == 'SAME':
        OH, pt, _ = same_pad(H, kh, sh)
        OW, pl, _ = same_pad(W, kw, sw)
    else:
        pt = pl = layer.pad_int
        OH = (H + 2 * pt - kh) // sh + 1
        OW = (W + 2 * pl - kw) // sw + 1
    return (N, H, W, Cin, Cout, kh, kw, sh, sw, pt, pl, OH, OW)


def _conv_xkind(layer, geom):
    """Mantissa type of the conv input (F7/H2): s8 up to 8 bits; the 9-bit activations are u8 when the input is
    known non-negative, the {hi,hi,lo,0} x 16 split for a signed 3-channel image, else s16 hi|hi|lo."""
    N, H, W, Cin, Cout, kh, kw = geom[:7]
    xb = layer.qX.bits
    if layer.qW.bits > 8 or xb > 16:
        raise _lib.LbtError('Conv2d_q: weights wider than 8 bits need the hi/lo GEMM split (not built yet)')
    if xb <= 8:
        return Q.MANT_S8
    if xb <= 9 and not layer.input_signed:
        return Q.MANT_U8
    if xb <= 9 and Cin == 3 and layer.implicit and kh * kw * 16 <= 65536 and _implicit_ok(Cout, 1, 1):
        return Q.MANT_S9C3
    return Q.MANT_S16


def _conv_quantize_input(layer, x, geom):
    """Xq of dfxp:287 as mantissas.  Uses the mantissas a fused producer already made with this very quantiser
    (``x._lbt_q``, see conv_bn_unit) when there are any."""
    xkind = _conv_xkind(layer, geom)
    pre = getattr(x, '_lbt_q', None)
    if pre is not None and id(layer.qX) in pre:
        xm, kind = pre[id(layer.qX)]
        assert kind == xkind, (kind, xkind)
        return xm, xkind
    if getattr(x, '_lbt_hollow', False):
        raise _lib.LbtError('Conv2d_q: got a mantissa-only activation made for a different quantiser')
    N, H, W = geom[:3]
    x_nhwc = _mem_contig(x).permute(0, 2, 3, 1)
    if xkind == Q.MANT_S9C3:
        xm = torch.empty(N, H, W, 16, dtype=torch.int8, device=x.device)
        layer.qX.quantize(x_nhwc, want_fp32=False, mant_kind=xkind, out_mant=xm)
        return xm, xkind
    _, xm = layer.qX.quantize(x_nhwc, want_fp32=False, mant_kind=xkind)
    return xm, xkind


def _stem_applies(geom):
    """Shapes lbt_conv_i8_wgrad_c3 takes (the 7x7/2 ImageNet stem): stride 2, <= 8 x 8 taps, 64 filters, even H."""
    N, H, W, Cin, Cout, kh, kw, sh, sw = geom[:9]
    return STEM_WGRAD and sh == 2 and sw == 2 and kh <= 8 and kw <= 8 and Cout == 64 and H % 2 == 0


def _stem_work(layer, geom, dev):
    N, H, OW = geom[0], geom[1], geom[12]
    nb = int(_lib.lib().lbt_stem_pack8_bytes(N, H, OW))
    work = getattr(layer, '_stem_work8', None)
    if work is None or work.numel() != nb or work.device != torch.device(dev):
        work = layer._stem_work8 = torch.empty(nb, dtype=torch.int8, device=dev)
        layer._stem_packed = False
    return work, nb


def _stem_prepack(layer, xm, xkind, geom):
    """Forward pass of a first convolution inside a Trainer step: re-pack the image for lbt_conv_i8_wgrad_c3 NOW, on the side
    stream beside the convolution, instead of at the very end of the step in front of the weight-gradient kernel."""
    rt = layer.qX.runtime
    if (xkind != Q.MANT_S9C3 or not _stem_applies(geom) or not torch.is_grad_enabled() or not layer.weight.requires_grad or
            not (rt.overlap and rt._arena_on and rt.grad_sink is not None and rt.grad_sink.active and _lib.profiler is None)):
        return
    N, H, W = geom[:3]
    dev = xm.device
    work, _ = _stem_work(layer, geom, dev)
    main, side = torch.cuda.current_stream(dev), rt.side_stream(dev)
    side.wait_stream(main)
    with torch.cuda.stream(side):
        layer._stem_packed = _lib.try_call('lbt_stem_pack8', _lib.ptr(xm), N, H, W, geom[12], geom[10], _lib.ptr(work), _lib.stream(),
                                           meta=dict(bytes=N * H * W * 16 + work.numel()))
    xm.record_stream(side)
    rt._side_pending = True


def _flush_head_beside(rt, fork, main, side):
    """Backward of the FIRST layer, before its weight-gradient kernel goes to the side stream: every gradient collected so far
    is finalised on the main stream (which has nothing else left) while that last kernel runs (GradSink.flush_head)."""
    sink = rt.grad_sink
    if sink is None or not sink.active:
        return
    if fork:
        ev = torch.cuda.Event()
        ev.record(side)                      # every earlier weight-gradient kernel
        with torch.cuda.stream(main):
            main.wait_event(ev)
            sink.flush_head()
    else:
        sink.flush_head()


def _conv_params(layer, weight, bias):
    """(prep entry or None, weight mantissas or None, quantised bias or None) for this step."""
    if not weight.is_contiguous():      # HWIO memory order is part of the semantics (noise broadcasts over kh)
        weight = weight.contiguous()
    prep = _prepared(layer)
    bq = wm = None
    if prep is None:
        _, wm = layer.qW.quantize(weight, want_fp32=False, mant_kind=Q.MANT_S8)               # dfxp:289
        if bias is not None:
            bq, _ = layer.qb.quantize(bias)                                                    # dfxp:294
    else:
        bq = prep.get('bq')
    return prep, wm, bq


def _conv_fprop(layer, geom, xm, xkind, prep, wm, bq, out2d, bnq=None):
    """dfxp:291-296 on mantissas: out2d (fp32 [M, Cout]) or, with ``bnq``, the fused quantise + statistics epilogue."""
    N, H, W, Cin, Cout, kh, kw, sh, sw, pt, pl, OH, OW = geom
    e = -(layer.qX.bits - 1) - (layer.qW.bits - 1)
    Kf = kh * kw * Cin
    ibx, ibw = layer.qX.range, layer.qW.range
    if xkind == Q.MANT_S9C3:
        if prep is not None:
            wt = prep['wt']
        else:
            w3 = wm.view(kh * kw, 3, Cout)
            w16 = torch.cat([w3, w3, w3, torch.zeros(kh * kw, 7, Cout, dtype=torch.int8, device=xm.device)], dim=1)
            wt = _transpose_bytes(w16.view(kh * kw * 16, Cout))
        _conv_implicit(xm, Q.MANT_S8, wt, Cout, kh, kw, sh, sw, pt, pl, OH, OW, ibx, ibw, e, bq, out2d, bnq)
        return
    segs = 3 if xkind == Q.MANT_S16 else 1
    wt = prep['wt'] if prep is not None else _transpose_bytes(wm.view(Kf, Cout))     # B operand [Cout, Kf]
    if segs == 3:
        wt = _as_operand(torch.cat([wt, wt, wt], dim=1))
    gbnq = None if bnq is None else (bnq[0], bnq[1], bnq[2], OH * OW)
    if kh == 1 and kw == 1 and sh == 1 and sw == 1 and segs == 1 and Cin % 16 == 0 and pt == 0 and pl == 0:
        G.gemm_i8(xm.reshape(N * H * W, Cin), wt, ibA=ibx, ibB=ibw, exp_const=e, bias=bq, out=out2d, bnq=gbnq)   # 1x1
    elif layer.implicit and segs == 1 and _implicit_ok(Cin, kh, kw):
        _conv_implicit(xm, xkind, wt, Cout, kh, kw, sh, sw, pt, pl, OH, OW, ibx, ibw, e, bq, out2d, bnq)     # dfxp:291
    else:
        A = _im2col(xm, xkind, OH, OW, kh, kw, sh, sw, pt, pl, False)
        G.gemm_i8(A, wt, ibA=ibx, ibB=ibw, exp_const=e, bias=bq, out=out2d, bnq=gbnq)


def _conv_backward(layer, geom, xm, xkind, wm, prep, gm, need_dx, need_dw, need_db, addend=None, shortcut=None):
    """dfxp:302-305 from the quantised gradient mantissas gm [N, OH, OW, Cout] (s8): (dX NHWC fp32, dW, db).
    ``addend`` (NHWC fp32, the shape of dX): the gradient reaching the same input along another branch (residual
    shortcut), added in the dgrad epilogue instead of by a separate pass over the tensor.  ``shortcut``: a strided block's
    1x1 shortcut parked by _BlockDgrad (only with the parity-class path, see _block_dgrad_ok): its input gradient is computed
    in the same launch as this one (lbt_conv_i8_dgrad_block), or first on its own and then added as ``addend``."""
    N, H, W, Cin, Cout, kh, kw, sh, sw, pt, pl, OH, OW = geom
    xb, wb, gb = layer.qX.bits, layer.qW.bits, layer.qG.bits
    dev = gm.device
    M = N * OH * OW
    g2 = gm.view(M, Cout)
    Kf = kh * kw * Cin
    dW = db = dx = None
    rt = layer.qX.runtime
    # ---- wgrad: dW[Kf, Cout] = A^T[Kf, M] . G[M, Cout], reduction over M split across the SMs.  It shares only its
    # inputs with dgrad, so (inside a Trainer step) it runs on a side stream: a parallel branch of the step's graph ----
    fork = need_dw and rt.overlap and rt._arena_on and rt.grad_sink is not None and rt.grad_sink.active and _lib.profiler is None
    main = torch.cuda.current_stream(dev) if fork else None
    side = rt.side_stream(dev) if fork else None
    if fork:
        side.wait_stream(main)
    if need_dw:
      with (torch.cuda.stream(side) if fork else contextlib.nullcontext()):
          acc = rt.zeros_i64(Kf * Cout, dev).view(Kf, Cout)
          at = gt = None
          if xkind == Q.MANT_S9C3:
              if not _implicit_ok(Cout, 1, 1):
                  raise _lib.LbtError('first-layer implicit wgrad needs Cout in {16,32,64} or a multiple of 128')
              done = False
              _flush_head_beside(rt, fork, main, side)
              if _stem_applies(geom):
                  # the 7x7/2 ImageNet stem: 8-byte pixels {hi, 0, lo, 0}, one tiled TMA load per filter row (conv_stem.cu);
                  # dW[r, s, c] = 2 * acc8[r, s, c] + acc8[r, s, 4 + c]
                  work, nb = _stem_work(layer, geom, dev)
                  repack = 0 if getattr(layer, '_stem_packed', False) else 1       # 0: _stem_prepack ran in the forward pass
                  layer._stem_packed = False
                  acc8 = rt.zeros_i64(512 * Cout, dev)
                  done = _lib.try_call('lbt_conv_i8_wgrad_c3', _lib.ptr(xm), N, H, W, _lib.ptr(g2), Q.MANT_S8, Cout, kh, kw, pt, pl,
                                       OH, OW, _lib.ptr(work), repack, _lib.ptr(acc8), 1, _lib.stream(),
                                       meta=dict(ops=2 * M * Cout * Kf, bytes=N * H * W * 16 + nb + M * Cout + 8 * 512 * Cout))
                  if done:
                      a = acc8.view(8, 8, 8, Cout)[:kh, :kw]
                      acc = (2 * a[:, :, 0:3] + a[:, :, 4:7]).reshape(Kf, Cout).contiguous()
              if not done:
                  # 16 pseudo-channels {hi, hi, lo, 0}: dW[c] = acc[hi c] + acc[hi' c] + acc[lo c]  (k = 2*hi + lo)
                  acc16 = rt.zeros_i64(kh * kw * 16 * Cout, dev).view(kh * kw * 16, Cout)
                  _lib.call('lbt_conv_i8_wgrad', _lib.ptr(xm), Q.MANT_S8, N, H, W, 16, _lib.ptr(g2), Q.MANT_S8, Cout, kh, kw,
                            sh, sw, pt, pl, OH, OW, _lib.ptr(acc16), 1, 0, _lib.stream(),
                            meta=dict(ops=2 * M * Cout * Kf, bytes=N * H * W * 16 + M * Cout + 8 * kh * kw * 16 * Cout))
                  a = acc16.view(kh * kw, 16, Cout)
                  acc = (a[:, 0:3] + a[:, 3:6] + a[:, 6:9]).reshape(Kf, Cout).contiguous()
          elif layer.implicit and xkind != Q.MANT_S16 and _implicit_ok(Cin, kh, kw) and _implicit_ok(Cout, 1, 1):
              # implicit wgrad: X blocks and G blocks feed the tensor cores MN-major, no transposes
              _lib.call('lbt_conv_i8_wgrad', _lib.ptr(xm), xkind, N, H, W, Cin, _lib.ptr(g2), Q.MANT_S8, Cout, kh, kw,
                        sh, sw, pt, pl, OH, OW, _lib.ptr(acc), 1, 0, _lib.stream(),
                        meta=dict(ops=2 * M * Cout * Kf, bytes=N * H * W * Cin + M * Cout + 8 * Kf * Cout))
          else:
              gt = _transpose_bytes(g2)                                                       # [Cout, M]
              A = _im2col(xm, xkind, OH, OW, kh, kw, sh, sw, pt, pl, False)
              at = _transpose_bytes(A)                                                        # [Kf*segs, M]
          if at is None:
              pass
          elif xkind == Q.MANT_S16:
              G.gemm_i8_acc64(at[:Kf], gt, acc, alpha=2)                                      # k = 2*hi + lo
              G.gemm_i8_acc64(at[2 * Kf:], gt, acc, alpha=1)
          else:
              G.gemm_i8_acc64(at, gt, acc, alpha=1)
          dW = _emit_grad(rt, layer.weight, acc, ibA=layer.qX.range, ibB=layer.qG.range, exp_const=-(xb - 1) - (gb - 1),
                          add_scale=2 * layer.weight_decay, shape=(kh, kw, Cin, Cout))         # dfxp:302
    if need_db:
        db = _emit_grad(rt, layer.bias, _colsum(g2, Q.MANT_S8, rt), ibA=layer.qG.range, exp_const=-(gb - 1))      # dfxp:304
    # ---- dgrad: dX[NHW, Cin] = im2colT(G)[NHW, kh*kw*Cout] . Wt[Cin, kh*kw*Cout] ----
    if need_dx:
        K2 = kh * kw * Cout
        dx = torch.empty(N, H, W, Cin, dtype=torch.float32, device=dev)
        ad2 = addend.reshape(N * H * W, Cin) if addend is not None else None
        e = -(gb - 1) - (wb - 1)
        pw2 = prep['w2'] if prep is not None else None        # packed by lbt_param_prep in the form used below
        if prep is not None and pw2 is None:
            raise _lib.LbtError('Conv2d_q: no input gradient for a 3-channel first-layer convolution')
        if kh == 1 and kw == 1 and sh == 1 and sw == 1 and Cout % 16 == 0 and pt == 0 and pl == 0:
            w2 = pw2 if pw2 is not None else _as_operand(wm.view(Cin, Cout))
            G.gemm_i8(g2, w2, ibA=layer.qG.range, ibB=layer.qW.range, exp_const=e, out=dx.view(N * H * W, Cin), addend=ad2)
        elif layer.implicit and sh == 1 and sw == 1 and _implicit_ok(Cout, kh, kw):
            # stride 1: dX = conv(G, rot180(W)) with padding (k - 1 - pad): the same implicit-GEMM kernel
            w2 = pw2 if pw2 is not None else _as_operand(wm.flip(0, 1).permute(2, 0, 1, 3).reshape(Cin, K2))
            _conv_implicit(gm, Q.MANT_S8, w2, Cin, kh, kw, 1, 1, kh - 1 - pt, kw - 1 - pl, H, W, layer.qG.range,
                           layer.qW.range, e, None, dx.view(N * H * W, Cin), addend=ad2)   # dfxp:305
        elif layer.implicit and _gather_ok(Cout, Cin, kh, kw) and sh <= 4 and sw <= 4:
            # any stride: the transposed gather runs in the kernel's loader warps (lbt_conv_i8_dgrad), no im2col matrix
            w2 = pw2 if pw2 is not None else _as_operand(wm.view(kh * kw, Cin, Cout).permute(1, 0, 2).reshape(Cin, K2))
            _lib.call('lbt_conv_i8_dgrad', _lib.ptr(gm), Q.MANT_S8, N, OH, OW, Cout, _lib.ptr(w2), Q.MANT_S8, w2.stride(0),
                      Cin, kh, kw, sh, sw, pt, pl, H, W, _lib.ptr(layer.qG.range), _lib.ptr(layer.qW.range), int(e),
                      _lib.ptr(dx), Cin, _lib.ptr(ad2), _lib.stream(),
                      meta=dict(ops=2 * N * H * W * Cin * K2, bytes=N * OH * OW * Cout + Cin * K2 + N * H * W * Cin * 4))
        elif (prep['classes'] if prep is not None else _dgrad_classes_ok(layer, Cin, Cout, kh, kw, sh, sw)):
            # wide gathered channels: one stride-1 sub-convolution per parity class of input pixels, no im2col matrix
            if pw2 is not None:
                w2 = pw2
            else:
                perm = torch.tensor(_class_perm(kh, kw, sh, sw), device=dev)
                w2 = _as_operand(wm.view(kh * kw, Cin, Cout).index_select(0, perm).permute(1, 0, 2).reshape(Cin, K2))
            done = shortcut is not None and addend is None and _dgrad_block(layer, geom, gm, w2, e, dx, shortcut)
            if not done:
                if shortcut is not None:      # the kernel declined the shapes: the shortcut's dgrad first, then this one adds it
                    ad2 = _shortcut_dgrad(shortcut).reshape(N * H * W, Cin)
                _lib.call('lbt_conv_i8_dgrad_strided', _lib.ptr(gm), Q.MANT_S8, N, OH, OW, Cout, _lib.ptr(w2), Q.MANT_S8,
                          w2.stride(0), Cin, kh, kw, sh, sw, pt, pl, H, W, _lib.ptr(layer.qG.range), _lib.ptr(layer.qW.range), int(e),
                          _lib.ptr(dx), Cin, _lib.ptr(ad2), _lib.stream(),
                          meta=dict(ops=2 * N * OH * OW * Cin * K2,
                                    bytes=N * OH * OW * Cout * min(sh * sw, kh * kw) + Cin * K2 + N * H * W * Cin * 4))
        else:
            w2 = pw2 if pw2 is not None else _as_operand(wm.view(kh * kw, Cin, Cout).permute(1, 0, 2).reshape(Cin, K2))
            A2 = _im2col(gm, Q.MANT_S8, H, W, kh, kw, sh, sw, pt, pl, True)
            G.gemm_i8(A2, w2, ibA=layer.qG.range, ibB=layer.qW.range, exp_const=e, out=dx.view(N * H * W, Cin), addend=ad2)
    if fork:
        # NO join here: the weight gradient is needed only by the end-of-backward finalize (Runtime.join_side, called by
        # the Trainer before lbt_finalize_multi), so it overlaps the rest of the backward chain.  Its operands must not
        # be recycled by the allocator before the side stream is done with them.
        for t in (xm, gm):
            t.record_stream(side)
        rt._side_pending = True
    return dx, dW, db


FUSE_BLOCK_DGRAD = os.environ.get('LBT_FUSE_BLOCK_DGRAD', '1') != '0'   # module switch: a downsampling block's input gradient (every
                      # parity class of its strided convolution and its 1x1 shortcut) in one launch, lbt_conv_i8_dgrad_block
_block_dgrad_count = 0   # lbt_conv_i8_dgrad_block launches (tests)


class _BlockDgrad:
    """Backward hand-off between the two units of a downsampling block that read the same input: the first unit of the residual
    branch (a strided convolution, which hands its input to the shortcut as an alias) and the 1x1 shortcut unit.  The shortcut
    unit runs its batch-norm backward and weight gradient as usual, then parks its gradient mantissas here and returns a shape
    carrier for dX; the alias returns it to the first unit, whose input-gradient launch then writes the sum of both branches
    (lbt_conv_i8_dgrad_block).  The fp32 shortcut gradient is never written."""

    def __init__(self):
        self.armed = False     # the first unit hands its input to the shortcut through the alias (set in its forward)
        self.parked = None     # (layer, geom, xkind, wm, prep, gm) of the shortcut

    def take(self):
        p, self.parked = self.parked, None
        return p


def _block_dgrad_ok(layer, geom, prep):
    """The first unit's input gradient takes the parity-class path, where lbt_conv_i8_dgrad_block applies."""
    N, H, W, Cin, Cout, kh, kw, sh, sw, pt, pl, OH, OW = geom
    if (sh, sw) == (1, 1) or layer.qG.bits > 8:
        return False
    if layer.implicit and _gather_ok(Cout, Cin, kh, kw) and sh <= 4 and sw <= 4:
        return False
    return bool(prep['classes'] if prep is not None else _dgrad_classes_ok(layer, Cin, Cout, kh, kw, sh, sw))


def _shortcut_dgrad(parked):
    """The parked shortcut's input gradient on its own (NHWC fp32), as its unit would have computed it."""
    layer, geom, xkind, wm, prep, gm = parked
    dx, _, _ = _conv_backward(layer, geom, None, xkind, wm, prep, gm, True, False, False)
    return dx


def _dgrad_block(layer, geom, gm, w2, e, dx, shortcut):
    """lbt_conv_i8_dgrad_block: dx = this strided convolution's input gradient + the parked shortcut's, in one launch.
    False when the kernel does not take the shapes (the caller then runs the two launches)."""
    global _block_dgrad_count
    N, H, W, Cin, Cout, kh, kw, sh, sw, pt, pl, OH, OW = geom
    sl, sgeom, _, swm, sprep, sgm = shortcut
    sN, sH, sW, sCin, sCout, skh, skw, ssh, ssw, spt, spl, sOH, sOW = sgeom
    if (sN, sH, sW, sCin) != (N, H, W, Cin) or (skh, skw, ssh, ssw, spt, spl) != (1, 1, sh, sw, 0, 0):
        return False
    spw2 = sprep['w2'] if sprep is not None else None
    sw2 = spw2 if spw2 is not None else _as_operand(swm.view(Cin, sCout))
    se = -(sl.qG.bits - 1) - (sl.qW.bits - 1)
    K2 = kh * kw * Cout
    done = _lib.try_call('lbt_conv_i8_dgrad_block', _lib.ptr(gm), Q.MANT_S8, N, OH, OW, Cout, _lib.ptr(w2), Q.MANT_S8,
                         w2.stride(0), Cin, kh, kw, sh, sw, pt, pl, H, W,
                         _lib.ptr(layer.qG.range), _lib.ptr(layer.qW.range), int(e), _lib.ptr(sgm), Q.MANT_S8, sOH, sOW, sCout,
                         _lib.ptr(sw2), Q.MANT_S8, sw2.stride(0),
                         _lib.ptr(sl.qG.range), _lib.ptr(sl.qW.range), int(se), _lib.ptr(dx), Cin, None, _lib.stream(),
                         meta=dict(ops=2 * N * OH * OW * Cin * K2 + 2 * N * sOH * sOW * Cin * sCout,
                                   bytes=N * OH * OW * Cout + N * sOH * sOW * sCout + Cin * (K2 + sCout) + N * H * W * Cin * 4))
    if done:
        _block_dgrad_count += 1
    return done


def _check_layer_bits(who, bits, grad_bits):
    """Widths the tensor-core layers take, checked at construction (the reference's --bits is free, main.py:112; the
    quantiser itself — lbt_quantize / weight_quantization — takes every width of dfxp:21): weights and activations ride the
    8-bit integer tensor cores (conv activations bits+1 = 9 as u8 / split), gradients up to 16 bits as hi/lo halves."""
    if not 2 <= int(bits) <= 8:
        raise _lib.LbtError('%s: bits=%d — the integer tensor-core layers take 2..8-bit weights/activations '
                            '(gradients up to 16 bits via grad_bits); wider DFXP only through weight_quantization()' % (who, bits))
    if grad_bits is not None and not 2 <= int(grad_bits) <= 16:
        raise _lib.LbtError('%s: grad_bits=%d — gradient quantisers take 2..16 bits' % (who, grad_bits))


def _split16(gm16):
    """s16 mantissas -> (hi s8, lo u8) with k = 256*hi + lo (lbt_split_s16)."""
    hi = torch.empty(gm16.shape, dtype=torch.int8, device=gm16.device)
    lo = torch.empty(gm16.shape, dtype=torch.uint8, device=gm16.device)
    _lib.call('lbt_split_s16', _lib.ptr(gm16), gm16.numel(), _lib.ptr(hi), _lib.ptr(lo), _lib.stream(),
              meta=dict(bytes=gm16.numel() * 4))
    return hi, lo


def _conv_backward16(layer, geom, xm, xkind, wm, prep, hi, lo, need_dx, need_dw, need_db, gm16=None, addend=None):
    """dfxp:302-305 with a gradient quantiser wider than 8 bits (BASELINE config 5: 16-bit G).  The gradient mantissas arrive
    as their two byte planes k = 256*hi + lo (hi s8, lo u8; written directly by lbt_bn_bwd_apply in the fused units, by
    lbt_split_s16 otherwise).  wgrad: every product runs twice on the 8-bit tensor cores, alpha = 256 / 1 into the exact
    int64 accumulators.  dgrad: ONE launch of lbt_gemm_i8_dual — both planes against one copy of the filter, two accumulators
    in tensor memory combined before the single rounding — so dX is RN_fp32(exact integer dot * 2^e) with no int64 tensor in
    HBM.  ``addend``: the gradient of the other branch (residual shortcut), added in the dgrad epilogue."""
    N, H, W, Cin, Cout, kh, kw, sh, sw, pt, pl, OH, OW = geom
    xb, wb, gb = layer.qX.bits, layer.qW.bits, layer.qG.bits
    dev = hi.device
    M = N * OH * OW
    Kf = kh * kw * Cin
    rt = layer.qX.runtime
    halves = ((hi, Q.MANT_S8, 256), (lo, Q.MANT_U8, 1))
    dW = db = dx = None
    fork = need_dw and rt.overlap and rt._arena_on and rt.grad_sink is not None and rt.grad_sink.active and _lib.profiler is None
    main = torch.cuda.current_stream(dev) if fork else None
    side = rt.side_stream(dev) if fork else None
    if fork:
        side.wait_stream(main)
    if need_dw:
      with (torch.cuda.stream(side) if fork else contextlib.nullcontext()):
        acc = rt.zeros_i64(Kf * Cout, dev).view(Kf, Cout)
        if xkind == Q.MANT_S9C3:
            if not _implicit_ok(Cout, 1, 1):
                raise _lib.LbtError('first-layer implicit wgrad needs Cout in {16,32,64} or a multiple of 128')
            done = False
            _flush_head_beside(rt, fork, main, side)
            if _stem_applies(geom):
                # the 7x7/2 ImageNet stem (conv_stem.cu): both byte planes against ONE re-packed copy of the image
                work, nb = _stem_work(layer, geom, dev)
                repack = 0 if getattr(layer, '_stem_packed', False) else 1       # 0: _stem_prepack ran in the forward pass
                layer._stem_packed = False
                acc8 = rt.zeros_i64(512 * Cout, dev)
                done = True
                for i, (g_, kind, alpha) in enumerate(halves):
                    done = done and _lib.try_call('lbt_conv_i8_wgrad_c3', _lib.ptr(xm), N, H, W, _lib.ptr(g_), kind, Cout, kh, kw, pt,
                                                  pl, OH, OW, _lib.ptr(work), repack if i == 0 else 0, _lib.ptr(acc8), alpha, _lib.stream(),
                                                  meta=dict(ops=M * Cout * Kf, bytes=(N * H * W * 16 + nb if i == 0 else 0) + nb + M * Cout))
                if done:
                    a = acc8.view(8, 8, 8, Cout)[:kh, :kw]
                    acc = (2 * a[:, :, 0:3] + a[:, :, 4:7]).reshape(Kf, Cout).contiguous()
            if not done:
                acc16 = rt.zeros_i64(kh * kw * 16 * Cout, dev).view(kh * kw * 16, Cout)
                for g_, kind, alpha in halves:
                    _lib.call('lbt_conv_i8_wgrad', _lib.ptr(xm), Q.MANT_S8, N, H, W, 16, _lib.ptr(g_), kind, Cout, kh, kw, sh, sw,
                              pt, pl, OH, OW, _lib.ptr(acc16), alpha, 0, _lib.stream(),
                              meta=dict(ops=M * Cout * Kf, bytes=N * H * W * 16 + M * Cout + 8 * kh * kw * 16 * Cout))
                a = acc16.view(kh * kw, 16, Cout)
                acc = (a[:, 0:3] + a[:, 3:6] + a[:, 6:9]).reshape(Kf, Cout).contiguous()
        elif layer.implicit and xkind != Q.MANT_S16 and _implicit_ok(Cin, kh, kw) and _implicit_ok(Cout, 1, 1):
            # both byte planes in ONE launch (two accumulators, the input blocks loaded once, one atomic per element) ...
            done = DUAL_WGRAD and _lib.try_call('lbt_conv_i8_wgrad_dual', _lib.ptr(xm), xkind, N, H, W, Cin, _lib.ptr(hi), _lib.ptr(lo),
                                                Cout, kh, kw, sh, sw, pt, pl, OH, OW, _lib.ptr(acc), 1, 0, _lib.stream(),
                                                meta=dict(ops=2 * M * Cout * Kf, bytes=N * H * W * Cin + 2 * M * Cout + 8 * Kf * Cout))
            for g_, kind, alpha in (() if done else halves):      # ... else one pass per plane (alpha = 256 | 1)
                _lib.call('lbt_conv_i8_wgrad', _lib.ptr(xm), xkind, N, H, W, Cin, _lib.ptr(g_), kind, Cout, kh, kw, sh, sw,
                          pt, pl, OH, OW, _lib.ptr(acc), alpha, 0, _lib.stream(),
                          meta=dict(ops=M * Cout * Kf, bytes=N * H * W * Cin + M * Cout + 8 * Kf * Cout))
        else:
            A = _im2col(xm, xkind, OH, OW, kh, kw, sh, sw, pt, pl, False)
            at = _transpose_bytes(A)
            for g_, kind, alpha in halves:
                gt = _transpose_bytes(g_.view(M, Cout))
                if xkind == Q.MANT_S16:
                    G.gemm_i8_acc64(at[:Kf], gt, acc, alpha=2 * alpha)
                    G.gemm_i8_acc64(at[2 * Kf:], gt, acc, alpha=alpha)
                else:
                    G.gemm_i8_acc64(at, gt, acc, alpha=alpha)
        dW = _emit_grad(rt, layer.weight, acc, ibA=layer.qX.range, ibB=layer.qG.range, exp_const=-(xb - 1) - (gb - 1),
                        add_scale=2 * layer.weight_decay, shape=(kh, kw, Cin, Cout))
    if need_db:
        if gm16 is None:
            raise _lib.LbtError('Conv2d_q: the bias gradient of a 16-bit gradient needs the s16 mantissas')
        db = _emit_grad(rt, layer.bias, _colsum(gm16.view(M, Cout), Q.MANT_S16, rt), ibA=layer.qG.range, exp_const=-(gb - 1))
    if need_dx:
        K2 = kh * kw * Cout
        e = -(gb - 1) - (wb - 1)
        pw2 = prep['w2'] if prep is not None else None
        if prep is not None and pw2 is None:
            raise _lib.LbtError('Conv2d_q: no input gradient for a 3-channel first-layer convolution')
        dx = torch.empty(N, H, W, Cin, dtype=torch.float32, device=dev)
        ad2 = addend.reshape(N * H * W, Cin) if addend is not None else None
        one_by_one = kh == 1 and kw == 1 and sh == 1 and sw == 1 and Cout % 16 == 0 and pt == 0 and pl == 0
        rot = bool(prep is not None and prep.get('rot180'))
        done = False
        if one_by_one:
            w2 = pw2 if pw2 is not None else _as_operand(wm.view(Cin, Cout))
            a_hi, a_lo = hi.view(M, Cout), lo.view(M, Cout)
        elif rot:
            w2 = pw2                                      # rot180-packed: dX = conv(G, rot180 W), padding k - 1 - pad
            # both byte planes through the TMA halo kernel with two accumulators in tensor memory (no im2col matrices) where
            # the filter bank and two patches per ring slot fit (64 gathered channels); else im2col of both planes + dual GEMM
            done = DUAL_HALO and _lib.try_call(
                'lbt_conv_i8_fprop_dual', _lib.ptr(hi), _lib.ptr(lo), N, OH, OW, Cout, _lib.ptr(w2),
                Q.MANT_S8, w2.stride(0), Cin, kh, kw, kh - 1 - pt, kw - 1 - pl, H, W, _lib.ptr(layer.qG.range),
                _lib.ptr(layer.qW.range), int(e), _lib.ptr(dx), Cin, _lib.ptr(ad2), _lib.stream(),
                meta=dict(ops=2 * 2 * N * H * W * Cin * K2, bytes=2 * N * OH * OW * Cout + Cin * K2 + N * H * W * Cin * 4))
            if not done:
                a_hi = _im2col(hi, Q.MANT_S8, H, W, kh, kw, 1, 1, kh - 1 - pt, kw - 1 - pl, False)
                a_lo = _im2col(lo, Q.MANT_U8, H, W, kh, kw, 1, 1, kh - 1 - pt, kw - 1 - pl, False)
        elif prep is not None and prep.get('classes'):
            # strided layer: one dual-accumulator stride-1 sub-convolution per parity class (class-ordered filter from lbt_param_prep)
            _lib.call('lbt_conv_i8_dgrad_strided_dual', _lib.ptr(hi), _lib.ptr(lo), N, OH, OW, Cout, _lib.ptr(pw2), Q.MANT_S8,
                      pw2.stride(0), Cin, kh, kw, sh, sw, pt, pl, H, W, _lib.ptr(layer.qG.range), _lib.ptr(layer.qW.range), int(e),
                      _lib.ptr(dx), Cin, _lib.ptr(ad2), _lib.stream(),
                      meta=dict(ops=2 * 2 * N * OH * OW * Cin * K2, bytes=2 * N * OH * OW * Cout * min(sh * sw, kh * kw) + Cin * K2 + N * H * W * Cin * 4))
            done = True
        else:
            w2 = pw2 if pw2 is not None else _as_operand(wm.view(kh * kw, Cin, Cout).permute(1, 0, 2).reshape(Cin, K2))
            a_hi = _im2col(hi, Q.MANT_S8, H, W, kh, kw, sh, sw, pt, pl, True)
            a_lo = _im2col(lo, Q.MANT_U8, H, W, kh, kw, sh, sw, pt, pl, True)
        if not done:
            G.gemm_i8_dual(a_hi, a_lo, w2, ibA=layer.qG.range, ibB=layer.qW.range, exp_const=e, out=dx.view(N * H * W, Cin), addend=ad2)
    if fork:
        for t in (xm, hi, lo):
            t.record_stream(side)
        rt._side_pending = True
    return dx, dW, db


class _QConv2dFn(torch.autograd.Function):
    """dfxp:272-305 on integer mantissas: quantise X (bits+1), W, [b]; implicit GEMM fprop; in backward
    quantise the gradient, then wgrad (+2*wd*W), bias grad, dgrad."""

    @staticmethod
    def forward(ctx, x, weight, bias, layer):
        geom = _conv_geom(layer, x, weight)
        N, H, W, Cin, Cout, kh, kw, sh, sw, pt, pl, OH, OW = geom
        xm, xkind = _conv_quantize_input(layer, x, geom)                                       # dfxp:287
        prep, wm, bq = _conv_params(layer, weight, bias)
        _stem_prepack(layer, xm, xkind, geom)      # after _conv_params: that joined the parameter branch of the side stream
        y = torch.empty(N, OH, OW, Cout, dtype=torch.float32, device=x.device)
        _conv_fprop(layer, geom, xm, xkind, prep, wm, bq, y.view(N * OH * OW, Cout))
        ctx.layer, ctx.geom, ctx.xkind, ctx.prep = layer, geom, xkind, prep
        ctx.save_for_backward(xm, wm)
        return y.permute(0, 3, 1, 2)

    @staticmethod
    def backward(ctx, dy):
        layer = ctx.layer
        xm, wm = ctx.saved_tensors
        dy = _mem_contig(dy).permute(0, 2, 3, 1)
        needs = (ctx.needs_input_grad[0], ctx.needs_input_grad[1], layer.qb is not None and ctx.needs_input_grad[2])
        if layer.qG.bits > 8:                                                                  # 16-bit G: hi/lo split
            if layer.qG.bits > 16:
                raise _lib.LbtError('Conv2d_q: gradient quantisers wider than 16 bits are not supported')
            _, gm16 = layer.qG.quantize(dy, want_fp32=False, mant_kind=Q.MANT_S16)
            hi, lo = _split16(gm16)
            dx, dW, db = _conv_backward16(layer, ctx.geom, xm, ctx.xkind, wm, ctx.prep, hi, lo, *needs, gm16=gm16)
            return (dx.permute(0, 3, 1, 2) if dx is not None else None), dW, db, None
        _, gm = layer.qG.quantize(dy, want_fp32=False, mant_kind=Q.MANT_S8)                    # dfxp:300
        dx, dW, db = _conv_backward(layer, ctx.geom, xm, ctx.xkind, wm, ctx.prep, gm, ctx.needs_input_grad[0],
                                    ctx.needs_input_grad[1], layer.qb is not None and ctx.needs_input_grad[2])
        return (dx.permute(0, 3, 1, 2) if dx is not None else None), dW, db, None


class Conv2d_q(nn.Module):
    """Quantised 2-d convolution, dfxp:224-316 (``Conv2d_pq`` dfxp:129-221 is an identical copy).

    ``weight`` is stored HWIO like the reference's ``tf.Variable(ksize)``; ``padding`` is an int or
    'SAME' | 'VALID' with TensorFlow semantics.  ``input_signed=False`` declares a non-negative input
    (anything fed by a ReLU) so the bits+1 = 9-bit activation mantissas fit the u8 tensor-core type."""

    def __init__(self, bits, in_channels, out_channels, kernel_size, stride=1, padding='SAME', bias=True, *,
                 weight_decay=0.0, target_overflow_rate=0.0, input_range=2, weight_range=2, bias_range=2, grad_range=2,
                 grad_bits=None, input_signed=True, name='conv', runtime=None, implicit=True):
        super().__init__()
        rt = runtime or default_runtime()
        _check_layer_bits('Conv2d_q', bits, grad_bits)
        kh, kw = (kernel_size, kernel_size) if isinstance(kernel_size, int) else kernel_size
        self.stride = (stride, stride) if isinstance(stride, int) else tuple(stride)
        if isinstance(padding, str):
            assert padding in ('SAME', 'VALID')
            self.padding, self.pad_int = ('SAME', 0) if padding == 'SAME' else ('INT', 0)
        else:
            self.padding, self.pad_int = 'INT', int(padding)
        self.bits, self.weight_decay, self.input_signed, self.name = bits, float(weight_decay), input_signed, name
        self.implicit = implicit    # implicit-GEMM kernels where the shape allows; False = explicit im2col + GEMM
        self.fuse_bn = True         # may run as one unit with the BatchNorm2d_q that follows (conv_bn_unit)
        limit = (3 / (kh * kw * in_channels)) ** 0.5                                           # dfxp:247-254
        self.weight = nn.Parameter(torch.empty(kh, kw, in_channels, out_channels).uniform_(-limit, limit))
        self.bias = nn.Parameter(torch.zeros(out_channels)) if bias else None                  # dfxp:264
        # creation order = quantiser id order = the oracle's: X, W, [b], grad
        self.qX = QuantSite(rt, name + '/X', bits + 1, input_range, target_overflow_rate)      # dfxp:287 bits+1
        self.qW = QuantSite(rt, name + '/W', bits, weight_range, target_overflow_rate)
        self.qb = QuantSite(rt, name + '/b', bits, bias_range, target_overflow_rate) if bias else None
        self.qG = QuantSite(rt, name + '/grad', grad_bits or bits, grad_range, target_overflow_rate)

    def forward(self, x):
        return _QConv2dFn.apply(x, self.weight, self.bias, self)

    def info(self):
        return '%d bits conv2d: %dx%dx%d stride %dx%d pad %s weight_decay %f' % (
            self.bits, self.weight.shape[0], self.weight.shape[1], self.weight.shape[3], self.stride[0], self.stride[1],
            self.padding, self.weight_decay)


Conv2d_pq = Conv2d_q


# ------------------------------------------------------------------------------------------------
# Linear_q / Dense_q
# ------------------------------------------------------------------------------------------------


class _QLinearFn(torch.autograd.Function):
    """dfxp:384-393, 453-460: y = Q(X) @ Q(W) [+ Q(b)]; all three GEMMs on int8 mantissas."""

    @staticmethod
    def forward(ctx, x, weight, bias, layer):
        x = x.contiguous()
        Bsz, In = x.shape
        Out = weight.shape[1]
        if layer.qX.bits > 8 or layer.qW.bits > 8:
            raise _lib.LbtError('Linear_q: operands wider than 8 bits need the hi/lo GEMM split (not built yet)')
        _, xm = layer.qX.quantize(x, want_fp32=False, mant_kind=Q.MANT_S8)                     # dfxp:384 (bits)
        prep = _prepared(layer)
        bq = wm = None
        if prep is None:
            _, wm = layer.qW.quantize(weight, want_fp32=False, mant_kind=Q.MANT_S8)            # dfxp:386
            if bias is not None:
                bq, _ = layer.qb.quantize(bias)
            wt = _transpose_bytes(wm)                                                           # [Out, In]
        else:
            wt, bq = prep['wt'], prep.get('bq')
        y = G.gemm_i8(_as_operand(xm), wt, ibA=layer.qX.range, ibB=layer.qW.range,
                      exp_const=-(layer.qX.bits - 1) - (layer.qW.bits - 1), bias=bq)           # dfxp:388, 393
        ctx.layer, ctx.prep = layer, prep
        ctx.save_for_backward(xm, wm, weight)
        return y

    @staticmethod
    def backward(ctx, dy):
        layer = ctx.layer
        xm, wm, weight = ctx.saved_tensors
        xb, wb, gb = layer.qX.bits, layer.qW.bits, layer.qG.bits
        In, Out = weight.shape
        rt = layer.qX.runtime
        dX = dW = db = None
        if gb > 8:                                                                             # 16-bit G: hi/lo split
            if gb > 16:
                raise _lib.LbtError('Linear_q: gradient quantisers wider than 16 bits are not supported')
            _, gm16 = layer.qG.quantize(dy.contiguous(), want_fp32=False, mant_kind=Q.MANT_S16)
            hi, lo = _split16(gm16)
            halves = ((hi, 256), (lo, 1))
            if ctx.needs_input_grad[1]:
                acc = rt.zeros_i64(In * Out, dy.device).view(In, Out)
                xt = _transpose_bytes(xm)
                for g_, alpha in halves:
                    G.gemm_i8_acc64(xt, _transpose_bytes(g_), acc, alpha=alpha, k_splits=1)
                dW = _emit_grad(rt, layer.weight, acc, ibA=layer.qX.range, ibB=layer.qG.range,
                                exp_const=-(xb - 1) - (gb - 1), add_scale=2 * layer.weight_decay)
            if layer.qb is not None and ctx.needs_input_grad[2]:
                db = _emit_grad(rt, layer.bias, _colsum(gm16, Q.MANT_S16, rt), ibA=layer.qG.range, exp_const=-(gb - 1))
            if ctx.needs_input_grad[0]:
                w2 = ctx.prep['w2'] if ctx.prep is not None else _as_operand(wm)
                dX = G.gemm_i8_dual(_as_operand(hi), _as_operand(lo), w2, ibA=layer.qG.range, ibB=layer.qW.range,
                                    exp_const=-(gb - 1) - (wb - 1))                            # dfxp:460, one rounding
            return dX, dW, db, None
        _, gm = layer.qG.quantize(dy.contiguous(), want_fp32=False, mant_kind=Q.MANT_S8)       # dfxp:453
        if ctx.needs_input_grad[1]:
            acc = rt.zeros_i64(In * Out, dy.device).view(In, Out)
            G.gemm_i8_acc64(_transpose_bytes(xm), _transpose_bytes(gm), acc, alpha=1, k_splits=1)
            dW = _emit_grad(rt, layer.weight, acc, ibA=layer.qX.range, ibB=layer.qG.range,
                            exp_const=-(xb - 1) - (gb - 1), add_scale=2 * layer.weight_decay)  # dfxp:457
        if layer.qb is not None and ctx.needs_input_grad[2]:
            db = _emit_grad(rt, layer.bias, _colsum(gm, Q.MANT_S8, rt), ibA=layer.qG.range, exp_const=-(gb - 1))  # dfxp:459
        if ctx.needs_input_grad[0]:
            w2 = ctx.prep['w2'] if ctx.prep is not None else _as_operand(wm)
            dX = G.gemm_i8(_as_operand(gm), w2, ibA=layer.qG.range, ibB=layer.qW.range,
                           exp_const=-(gb - 1) - (wb - 1))                                     # dfxp:460
        return dX, dW, db, None


class Linear_q(nn.Module):
    """Quantised fully connected layer, dfxp:319-470 (``Dense_q``).  ``weight`` is [in, out]."""

    def __init__(self, bits, in_features, out_features, bias=True, *, weight_decay=0.0, target_overflow_rate=0.0,
                 input_range=2, weight_range=2, bias_range=2, grad_range=2, grad_bits=None, name='dense', runtime=None):
        super().__init__()
        rt = runtime or default_runtime()
        _check_layer_bits('Linear_q', bits, grad_bits)
        self.bits, self.weight_decay, self.name = bits, float(weight_decay), name
        limit = (6 / (in_features + out_features)) ** 0.5                                      # dfxp:338
        self.weight = nn.Parameter(torch.empty(in_features, out_features).uniform_(-limit, limit))
        self.bias = nn.Parameter(torch.zeros(out_features)) if bias else None
        self.qX = QuantSite(rt, name + '/X', bits, input_range, target_overflow_rate)          # dfxp:384: bits
        self.qW = QuantSite(rt, name + '/W', bits, weight_range, target_overflow_rate)
        self.qb = QuantSite(rt, name + '/b', bits, bias_range, target_overflow_rate) if bias else None
        self.qG = QuantSite(rt, name + '/grad', grad_bits or bits, grad_range, target_overflow_rate)

    def forward(self, x):
        return _QLinearFn.apply(x, self.weight, self.bias, self)

    def info(self):
        return '%d bits dense: %dx%d weight_decay %f' % (self.bits, self.weight.shape[0], self.weight.shape[1],
                                                        self.weight_decay)


Dense_q = Linear_q


# ------------------------------------------------------------------------------------------------
# BatchNorm: Normalization_q + Rescale_q
# ------------------------------------------------------------------------------------------------


class _WeightDecayGrad(torch.autograd.Function):
    """Adds 2*wd*p to the gradient of p (the reference keeps weight decay inside the layer's grad)."""

    @staticmethod
    def forward(ctx, p, wd):
        ctx.wd = wd
        ctx.save_for_backward(p)
        return p.view_as(p)

    @staticmethod
    def backward(ctx, g):
        (p,) = ctx.saved_tensors
        return g + (2 * ctx.wd) * p.detach(), None


class Normalization_q(nn.Module):
    """dfxp:539-623: quantise, batch moments of the QUANTISED input (biased variance), normalise;
    running statistics with momentum 0.999; backward quantises the gradient then applies the
    batch-norm VJP.  ``frozen`` (set by BatchNorm2d_q.freeze_statistics): in training mode too, normalise with the running
    statistics and leave them alone — the VJP is then g / sqrt(var + eps)."""

    def __init__(self, bits, num_features, momentum=0.999, eps=1e-5, *, target_overflow_rate=0.0, input_range=2,
                 grad_range=2, grad_bits=None, name='norm', runtime=None):
        super().__init__()
        rt = runtime or default_runtime()
        self.bits, self.momentum, self.eps, self.name = bits, momentum, eps, name
        self.register_buffer('X_mean_running', torch.zeros(num_features))                     # dfxp:565-568
        self.register_buffer('X_var_running', torch.ones(num_features))
        self.qX = QuantSite(rt, name + '/X', bits, input_range, target_overflow_rate)          # dfxp:584
        self.qG = QuantSite(rt, name + '/grad', grad_bits or bits, grad_range, target_overflow_rate)   # dfxp:621
        self.frozen = False

    def forward(self, x):
        x = _mem_contig(x)
        xq = _QuantSTE.apply(x, self.qX)
        axes = (0, 2, 3) if x.dim() == 4 else (0,)
        shape = (1, -1, 1, 1) if x.dim() == 4 else (1, -1)
        if self.training and not self.frozen:
            mean = xq.mean(dim=axes)                                                           # dfxp:588
            var = ((xq - mean.view(shape)) ** 2).mean(dim=axes)
            with torch.no_grad():                                                              # dfxp:602-612
                self.X_mean_running.mul_(self.momentum).add_((1 - self.momentum) * mean)
                self.X_var_running.mul_(self.momentum).add_((1 - self.momentum) * var)
        else:
            mean, var = self.X_mean_running, self.X_var_running
        y = (xq - mean.view(shape)) / ((var.view(shape) + self.eps) ** 0.5)                    # dfxp:616
        return _GradQuant.apply(y, self.qG)


class Rescale_q(nn.Module):
    """dfxp:626-694: y = Q(X) * Q(gamma) + Q(beta); weight decay on gamma (dfxp:689)."""

    def __init__(self, bits, num_features, *, weight_decay=0.0, target_overflow_rate=0.0, input_range=2, gamma_range=2,
                 beta_range=2, grad_range=2, grad_bits=None, name='rescale', runtime=None):
        super().__init__()
        rt = runtime or default_runtime()
        self.bits, self.weight_decay, self.name = bits, float(weight_decay), name
        self.gamma = nn.Parameter(torch.ones(num_features))
        self.beta = nn.Parameter(torch.zeros(num_features))
        self.qX = QuantSite(rt, name + '/X', bits, input_range, target_overflow_rate)          # dfxp:677
        self.qg = QuantSite(rt, name + '/g', bits, gamma_range, target_overflow_rate)          # dfxp:679
        self.qb = QuantSite(rt, name + '/b', bits, beta_range, target_overflow_rate)           # dfxp:681
        self.qG = QuantSite(rt, name + '/grad', grad_bits or bits, grad_range, target_overflow_rate)   # dfxp:687

    def forward(self, x):
        x = _mem_contig(x)
        shape = (1, -1, 1, 1) if x.dim() == 4 else (1, -1)
        xq = _QuantSTE.apply(x, self.qX)
        gq = _QuantSTE.apply(_WeightDecayGrad.apply(self.gamma, self.weight_decay), self.qg)
        bq = _QuantSTE.apply(self.beta, self.qb)
        y = xq * gq.view(shape) + bq.view(shape)                                               # dfxp:683
        return _GradQuant.apply(y, self.qG)


def _site_args(site, x_like):
    """(noise pointer tensor or None, Philox offset) of a quantiser site for the fused kernels."""
    rt = site.runtime
    if rt.noise_fn is not None:
        return rt.noise_fn(site, Q.rows_view(x_like)[1], x_like.device).contiguous(), 0
    return None, Q.make_offset(site.qid, 0)


def _to_mem(x):
    """Memory-order view of an activation: NHWC for logical-NCHW channels_last tensors, as is for 2-D."""
    x = _mem_contig(x)
    return x.permute(0, 2, 3, 1) if x.dim() == 4 else x


def _from_mem(t):
    return t.permute(0, 3, 1, 2) if t.dim() == 4 else t


def _bn_params(resc, gamma, beta):
    prep = _prepared(resc)
    if prep is not None:
        return prep['gq'], prep['bq']
    gq, _ = resc.qg.quantize(gamma.detach())                                                   # dfxp:679
    bq, _ = resc.qb.quantize(beta.detach())                                                    # dfxp:681
    return gq, bq


def _bn_fwd1(bn, xm_):
    """BN forward pass 1 on an fp32 memory-order tensor: (k1 s8, sums int64[2C])."""
    norm = bn[0]
    rt = norm.qX.runtime
    N, C = xm_.shape[0], xm_.shape[-1]
    n_inner = xm_.numel() // N
    sums = rt.zeros_i64(2 * C, xm_.device)
    k1 = torch.empty(xm_.shape, dtype=torch.int8, device=xm_.device)
    nz1, off1 = _site_args(norm.qX, xm_)
    _lib.call('lbt_bn_fwd_quant_stats', _lib.ptr(xm_), N, n_inner, C, norm.qX.bits, _lib.ptr(norm.qX.range),
              _lib.ptr(nz1), rt.seed, off1, _lib.ptr(rt.dev_step), _lib.ptr(k1), _lib.ptr(sums),
              _lib.ptr(norm.qX.counters), int(norm.qX.target == 0), _lib.stream(), meta=dict(bytes=xm_.numel() * 5))
    return k1, sums


def _bn_fwd2(bn, k1, sums, gq, bq, add_, relu, next_site=None, next_kind=Q.MANT_NONE, want_fp32=True, next2=None,
             running=False, want_k2=False):
    """BN forward pass 2 (+ residual add, ReLU, the consumer's input quantiser): (k2, out or None, next mantissas or None,
    relu_mode).  next2 = (site, kind): a second consumer's input quantiser; its mantissas come back as ``next2[2]`` (a list
    cell the caller passes in).  running: eval mode — normalise with the running statistics (``sums`` is not read, the
    running averages stay, k2 is None unless ``want_k2``: frozen statistics save it for lbt_bn_bwd_running)."""
    norm, resc = bn[0], bn[1]
    rt = norm.qX.runtime
    N, C = k1.shape[0], k1.shape[-1]
    n_inner = k1.numel() // N
    dev = k1.device
    k2 = torch.empty_like(k1) if (want_k2 or not running) else None
    out = torch.empty(k1.shape, dtype=torch.float32, device=dev) if want_fp32 else None
    nz2, off2 = _site_args(resc.qX, k1)
    relu_mode = 0 if not relu else (2 if add_ is not None else 1)
    qn = nm = None
    if next_site is not None:
        qn = next_site.abi(n_inner, dev)
        nm = torch.empty(k1.shape, dtype=torch.uint8 if next_kind == Q.MANT_U8 else torch.int8, device=dev)
    qn2 = nm2 = None
    if next2 is not None and qn is not None:
        site2, kind2 = next2[0], next2[1]
        qn2 = site2.abi(n_inner, dev)
        nm2 = torch.empty(k1.shape, dtype=torch.uint8 if kind2 == Q.MANT_U8 else torch.int8, device=dev)
        next2[2] = nm2
    nbytes = k1.numel() * ((1 if k2 is None else 2) + (4 if want_fp32 else 0) + (4 if add_ is not None else 0) +
                           (1 if nm is not None else 0) + (1 if nm2 is not None else 0))
    head = (_lib.ptr(k1), N, n_inner, C, norm.qX.bits, _lib.ptr(norm.qX.range))
    site = (float(norm.eps), resc.qX.bits, _lib.ptr(resc.qX.range), _lib.ptr(nz2), rt.seed, off2,
            _lib.ptr(rt.dev_step), _lib.ptr(resc.qX.counters), _lib.ptr(gq), _lib.ptr(bq), _lib.ptr(add_),
            1 if relu else 0, _lib.ptr(k2), _lib.ptr(out))
    nxt = (ctypes.addressof(qn) if qn is not None else None, _lib.ptr(nm), int(next_kind))
    nxt2 = (ctypes.addressof(qn2), _lib.ptr(nm2), int(next2[1])) if qn2 is not None else ()
    if running:
        _lib.call('lbt_bn_fwd_apply_running', *head, _lib.ptr(norm.X_mean_running), _lib.ptr(norm.X_var_running), *site,
                  int(resc.qX.target == 0), *nxt, *(nxt2 or (None, None, 0)), _lib.stream(), meta=dict(bytes=nbytes))
        return k2, out, nm, relu_mode
    args = head + (_lib.ptr(sums),) + site + (None, None, _lib.ptr(norm.X_mean_running), _lib.ptr(norm.X_var_running),
                                               float(norm.momentum), int(resc.qX.target == 0)) + nxt
    if nxt2:
        _lib.call('lbt_bn_fwd_apply2', *args, *nxt2, _lib.stream(), meta=dict(bytes=nbytes))
    else:
        _lib.call('lbt_bn_fwd_apply', *args, _lib.stream(), meta=dict(bytes=nbytes))
    return k2, out, nm, relu_mode


def _bn_backward(bn, g_, k1, k2, sums, gq, bq, out_, relu_mode, has_add, grad_site=None, want_dx=True):
    """Both BN backward passes on memory-order tensors: (dx fp32 or None, gradient mantissas of `grad_site` or None,
    dgamma, dbeta, d_add)."""
    norm, resc = bn[0], bn[1]
    rt = norm.qX.runtime
    N, C = k1.shape[0], k1.shape[-1]
    n_inner = k1.numel() // N
    dev = k1.device
    # [4C] sums; the two spare slots keep every later arena slice at the offset the step was tuned with (exactly 4C measured
    # 1.7 us slower on ResNet-20's 1.351 ms step, B200 at 1000 W)
    bsums = rt.zeros_i64(4 * C + 2, dev)
    d_add = torch.empty(k1.shape, dtype=torch.float32, device=dev) if has_add else None
    dx = torch.empty(k1.shape, dtype=torch.float32, device=dev) if want_dx else None
    # gradient quantisers wider than 8 bits (config 5: 16-bit G): kg1 travels as s16, and the convolution's gradient
    # mantissas leave the second pass as the two byte planes (hi s8, lo u8) its tensor-core kernels consume
    wide = max(resc.qG.bits, norm.qG.bits) > 8
    kg1_kind = Q.MANT_S16 if wide else Q.MANT_S8
    qg = gm = gm_lo = None
    if grad_site is not None:
        qg = grad_site.abi(n_inner, dev)
        gm = torch.empty_like(k1)
        if grad_site.bits > 8:
            gm_lo = torch.empty(k1.shape, dtype=torch.uint8, device=dev)
    kg1 = torch.empty(k1.shape, dtype=torch.int16 if wide else torch.int8, device=dev)
    nzg2, offg2 = _site_args(resc.qG, g_)
    nzg1, offg1 = _site_args(norm.qG, g_)
    _lib.call('lbt_bn_bwd_quant_stats', _lib.ptr(g_), _lib.ptr(out_), relu_mode, _lib.ptr(k2), _lib.ptr(k1), N, n_inner,
              C, resc.qX.bits, _lib.ptr(resc.qX.range), _lib.ptr(gq), _lib.ptr(bq), resc.qG.bits,
              _lib.ptr(resc.qG.range), _lib.ptr(nzg2), offg2, _lib.ptr(resc.qG.counters), norm.qG.bits,
              _lib.ptr(norm.qG.range), _lib.ptr(nzg1), offg1, _lib.ptr(norm.qG.counters), rt.seed,
              _lib.ptr(rt.dev_step), _lib.ptr(d_add), _lib.ptr(kg1), _lib.ptr(bsums),
              int(resc.qG.target == 0 and norm.qG.target == 0), kg1_kind, _lib.stream(),
              meta=dict(bytes=g_.numel() * (7 + (1 if wide else 0) + (4 if relu_mode == 2 else 0) + (4 if has_add else 0))))
    _lib.call('lbt_bn_bwd_apply', _lib.ptr(kg1), _lib.ptr(k1), N, n_inner, C, norm.qX.bits, _lib.ptr(norm.qX.range),
              _lib.ptr(sums), float(norm.eps), norm.qG.bits, _lib.ptr(norm.qG.range), _lib.ptr(bsums), _lib.ptr(dx),
              ctypes.addressof(qg) if qg is not None else None, _lib.ptr(gm), kg1_kind, _lib.ptr(gm_lo), _lib.stream(),
              meta=dict(bytes=k1.numel() * (2 + (1 if wide else 0) + (4 if want_dx else 0) + (1 if gm is not None else 0) +
                                            (1 if gm_lo is not None else 0))))
    # dbeta = sum gq2 (dfxp:690); dgamma = sum gq2 * xq2 + 2*wd*gamma (dfxp:689)
    dbeta = _emit_grad(rt, resc.beta, bsums[:C], ibA=resc.qG.range, exp_const=-(resc.qG.bits - 1))
    dgamma = _emit_grad(rt, resc.gamma, bsums[C:2 * C], ibA=resc.qG.range, ibB=resc.qX.range,
                        exp_const=-(resc.qG.bits - 1) - (resc.qX.bits - 1), add_scale=2 * resc.weight_decay)
    return dx, (gm if gm_lo is None else (gm, gm_lo)), dgamma, dbeta, d_add


def _bn_backward_frozen(bn, g_, k2, gq, bq, out_, relu_mode, has_add, grad_site=None, want_dx=True):
    """The BN backward pass of a layer with frozen statistics (BatchNorm2d_q.freeze_statistics), ONE launch
    (lbt_bn_bwd_running): mean and variance are constants, so dx = gq1 / sqrt(run_var + eps) needs neither k1 nor batch sums
    over the gradient.  Same results and return value as _bn_backward."""
    norm, resc = bn[0], bn[1]
    rt = norm.qX.runtime
    N, C = k2.shape[0], k2.shape[-1]
    n_inner = k2.numel() // N
    dev = k2.device
    bsums = rt.zeros_i64(2 * C, dev)
    d_add = torch.empty(k2.shape, dtype=torch.float32, device=dev) if has_add else None
    dx = torch.empty(k2.shape, dtype=torch.float32, device=dev) if want_dx else None
    qg = gm = gm_lo = None
    if grad_site is not None:
        qg = grad_site.abi(n_inner, dev)
        gm = torch.empty_like(k2)
        if grad_site.bits > 8:
            gm_lo = torch.empty(k2.shape, dtype=torch.uint8, device=dev)
    # any gradient quantiser wider than 8 bits (config 5: 16-bit G): the wide instantiation (64-bit partial sums, byte planes)
    wide = max(resc.qG.bits, norm.qG.bits, grad_site.bits if grad_site is not None else 0) > 8
    nzg2, offg2 = _site_args(resc.qG, g_)
    nzg1, offg1 = _site_args(norm.qG, g_)
    nbytes = k2.numel() * (5 + (4 if relu_mode == 2 else 0) + (4 if has_add else 0) + (4 if want_dx else 0) +
                           (1 if gm is not None else 0) + (1 if gm_lo is not None else 0))
    _lib.call('lbt_bn_bwd_running', _lib.ptr(g_), _lib.ptr(out_), relu_mode, _lib.ptr(k2), N, n_inner, C, resc.qX.bits,
              _lib.ptr(resc.qX.range), _lib.ptr(gq), _lib.ptr(bq), _lib.ptr(norm.X_var_running), float(norm.eps), resc.qG.bits,
              _lib.ptr(resc.qG.range), _lib.ptr(nzg2), offg2, _lib.ptr(resc.qG.counters), norm.qG.bits,
              _lib.ptr(norm.qG.range), _lib.ptr(nzg1), offg1, _lib.ptr(norm.qG.counters), rt.seed, _lib.ptr(rt.dev_step),
              _lib.ptr(d_add), _lib.ptr(bsums), _lib.ptr(dx), ctypes.addressof(qg) if qg is not None else None, _lib.ptr(gm),
              _lib.ptr(gm_lo), int(resc.qG.target == 0 and norm.qG.target == 0), Q.MANT_S16 if wide else Q.MANT_S8,
              _lib.stream(), meta=dict(bytes=nbytes))
    # dbeta = sum gq2 (dfxp:690); dgamma = sum gq2 * xq2 + 2*wd*gamma (dfxp:689)
    dbeta = _emit_grad(rt, resc.beta, bsums[:C], ibA=resc.qG.range, exp_const=-(resc.qG.bits - 1))
    dgamma = _emit_grad(rt, resc.gamma, bsums[C:2 * C], ibA=resc.qG.range, ibB=resc.qX.range,
                        exp_const=-(resc.qG.bits - 1) - (resc.qX.bits - 1), add_scale=2 * resc.weight_decay)
    return dx, (gm if gm_lo is None else (gm, gm_lo)), dgamma, dbeta, d_add


class _FusedBNFn(torch.autograd.Function):
    """Normalization_q + Rescale_q (+ residual add, + ReLU) in 2 forward and 2 backward passes over the
    activation (csrc/bn.cu), saving only the two s8 mantissa tensors for backward."""

    @staticmethod
    def forward(ctx, x, gamma, beta, add, bn, relu, running=False, frozen=False):
        # running: eval mode (or frozen statistics) without an autograd graph (BatchNorm2d_q._running); nothing is saved.
        # frozen: frozen statistics with a graph — the running-statistics forward, k2 saved for lbt_bn_bwd_running (no k1)
        x_ = _to_mem(x)
        k1, sums = _bn_fwd1(bn, x_)
        gq, bq = _bn_params(bn[1], gamma, beta)
        add_ = _to_mem(add) if add is not None else None
        k2, out, _, relu_mode = _bn_fwd2(bn, k1, sums, gq, bq, add_, relu, running=running or frozen, want_k2=frozen)
        if not running:
            ctx.bn, ctx.relu_mode, ctx.has_add, ctx.frozen = bn, relu_mode, add is not None, frozen
            ctx.save_for_backward(None if frozen else k1, k2, None if frozen else sums, gq, bq, out if relu_mode == 2 else None)
        return _from_mem(out)

    @staticmethod
    def backward(ctx, g):
        k1, k2, sums, gq, bq, out = ctx.saved_tensors
        if ctx.frozen:
            dx, _, dgamma, dbeta, d_add = _bn_backward_frozen(ctx.bn, _to_mem(g), k2, gq, bq, out, ctx.relu_mode, ctx.has_add)
        else:
            dx, _, dgamma, dbeta, d_add = _bn_backward(ctx.bn, _to_mem(g), k1, k2, sums, gq, bq, out, ctx.relu_mode, ctx.has_add)
        return _from_mem(dx), dgamma, dbeta, (_from_mem(d_add) if d_add is not None else None), None, None, None, None


class _ConvBNFn(torch.autograd.Function):
    """One Conv2d_q + BatchNorm2d_q unit (+ residual add, + ReLU) with every hand-off between the two modules kept
    in integer mantissas (north_star (2): the GEMM epilogue re-quantises its output, no fake-quant fp32 round trip):

      forward   X --Q_conv.X--> u8/s8 --tcgen05 conv, epilogue Q_norm.X + sum k, sum k^2--> k1 (s8)
                k1 --lbt_bn_fwd_apply--> k2 (s8, saved), out fp32 (only if wanted), mantissas for the NEXT conv
      backward  g --lbt_bn_bwd_quant_stats--> kg1 --lbt_bn_bwd_apply, epilogue Q_conv.grad--> gm (s8) --> wgrad, dgrad

    Same quantiser ids, ranges, noise streams and arithmetic as running the two modules one after the other:
    the results are bit-identical (tests/test_fused_gpu.py)."""

    @staticmethod
    def forward(ctx, x, weight, gamma, beta, add, conv, bn, relu, next_site, next_kind, want_fp32, alias, pool=None, next2=None,
                running=False, block=None, frozen=False):
        # running: eval mode (or frozen statistics) without an autograd graph (BatchNorm2d_q._running): the BN kernels normalise
        # with the running statistics, nothing is saved for backward.  frozen: frozen statistics while a graph is recorded —
        # the same kernels, k2 saved (k1 and the batch sums are not), backward through lbt_bn_bwd_running
        geom = _conv_geom(conv, x, weight)
        N, H, W, Cin, Cout, kh, kw, sh, sw, pt, pl, OH, OW = geom
        norm, resc = bn[0], bn[1]
        rt = norm.qX.runtime
        dev = x.device
        xm, xkind = _conv_quantize_input(conv, x, geom)                                        # dfxp:287
        prep, wm, _ = _conv_params(conv, weight, None)
        _stem_prepack(conv, xm, xkind, geom)       # after _conv_params: that joined the parameter branch of the side stream
        sums = rt.zeros_i64(2 * Cout, dev)
        k1 = torch.empty(N, OH, OW, Cout, dtype=torch.int8, device=dev)
        _conv_fprop(conv, geom, xm, xkind, prep, wm, None, None,
                    bnq=(norm.qX.abi(OH * OW * Cout, dev, arena=True), k1, sums))                          # dfxp:291 + :584-588
        gq, bq = _bn_params(resc, gamma, beta)
        add_ = _to_mem(add) if add is not None else None
        pooled = pidx = None
        if pool is not None and (add is not None or not FUSE_POOL_FWD or Cout != 64 or pool[:4] != (3, 2, 0, 0)):
            next_site, next_kind = None, Q.MANT_NONE        # next_site quantises the POOLED tensor: only the one-kernel path runs it
        if pool is not None and FUSE_POOL_FWD and add is None and Cout == 64 and pool[:4] == (3, 2, 0, 0):
            # the ImageNet stem: BN apply + ReLU + 3x3/2 max-pool in ONE kernel, the fp32 module output never exists
            pk, ps, ppt, ppl, POH, POW = pool
            k2 = None if running else torch.empty_like(k1)
            pooled = torch.empty(N, POH, POW, Cout, dtype=torch.float32, device=dev)
            pidx = torch.empty(N, POH, POW, Cout, dtype=torch.uint8, device=dev)
            nz2, off2 = _site_args(resc.qX, k1)
            qn = nmp = None
            if next_site is not None:
                qn = next_site.abi(POH * POW * Cout, dev)
                nmp = torch.empty(N, POH, POW, Cout, dtype=torch.uint8 if next_kind == Q.MANT_U8 else torch.int8, device=dev)
            head = (_lib.ptr(k1), N, OH, OW, Cout, norm.qX.bits, _lib.ptr(norm.qX.range))
            site = (float(norm.eps), resc.qX.bits, _lib.ptr(resc.qX.range), _lib.ptr(nz2), rt.seed, off2,
                    _lib.ptr(rt.dev_step), _lib.ptr(resc.qX.counters), _lib.ptr(gq), _lib.ptr(bq), 1 if relu else 0, _lib.ptr(k2))
            tail = (pk, ps, ppt, ppl, POH, POW, _lib.ptr(pooled), _lib.ptr(pidx),
                    ctypes.addressof(qn) if qn is not None else None, _lib.ptr(nmp), int(next_kind), _lib.stream())
            meta = dict(bytes=k1.numel() * (1 if running else 2) + pooled.numel() * (5 + (1 if nmp is not None else 0)))
            if running or frozen:
                done = _lib.try_call('lbt_bn_fwd_apply_running_pooled', *head, _lib.ptr(norm.X_mean_running),
                                     _lib.ptr(norm.X_var_running), *site, int(resc.qX.target == 0), *tail, meta=meta)
            else:
                done = _lib.try_call('lbt_bn_fwd_apply_pooled', *head, _lib.ptr(sums), *site, _lib.ptr(norm.X_mean_running),
                                     _lib.ptr(norm.X_var_running), float(norm.momentum), int(resc.qX.target == 0), *tail,
                                     meta=meta)
            if done:
                out, nm, relu_mode = None, nmp, (1 if relu else 0)
            else:
                pooled = pidx = None
                next_site, next_kind = None, Q.MANT_NONE
        if pooled is None:
            k2, out, nm, relu_mode = _bn_fwd2(bn, k1, sums, gq, bq, add_, relu, next_site, next_kind, True if pool is not None else want_fp32,
                                              next2=next2 if pool is None else None, running=running or frozen,
                                              want_k2=frozen)
        ctx.conv, ctx.bn, ctx.geom, ctx.xkind, ctx.prep = conv, bn, geom, xkind, prep
        ctx.relu_mode, ctx.has_add, ctx.frozen = relu_mode, add is not None, frozen
        # block: the downsampling block's _BlockDgrad; the unit with the alias is the first unit, the other one the shortcut
        ctx.block = None
        if block is not None and not running:
            if alias:       # only where the first unit's input gradient takes the parity-class path the kernel runs on
                block.armed = conv.qG.bits <= 8 and _block_dgrad_ok(conv, geom, prep)
                ctx.block = block if block.armed else None
            elif block.armed:
                ctx.block = block
        ctx.block_first = bool(alias)
        ctx.pool = None
        if pooled is not None:    # lbt_bn_fwd_apply_pooled did both
            ctx.pool = tuple(pool)
            out = pooled
        elif pool is not None:    # MaxPool_q behind the unit (ImageNet stem)
            pk, ps, ppt, ppl, POH, POW = pool
            pooled = torch.empty(N, POH, POW, Cout, dtype=torch.float32, device=dev)
            pidx = torch.empty(N, POH, POW, Cout, dtype=torch.uint8, device=dev)
            _lib.call('lbt_maxpool_fwd', _lib.ptr(out), N, OH, OW, Cout, pk, ps, ppt, ppl, POH, POW, _lib.ptr(pooled), _lib.ptr(pidx),
                      _lib.stream(), meta=dict(bytes=out.numel() * 4 + pooled.numel() * 5))
            ctx.pool = (pk, ps, ppt, ppl, POH, POW)
            out = pooled
        if not running:
            ctx.save_for_backward(xm, wm, None if frozen else k1, k2, None if frozen else sums, gq, bq,
                                  out if relu_mode == 2 else None, pidx)
        if out is None:       # mantissa-only activation: the fp32 tensor is never materialised (shape carrier only)
            out = torch.empty(1, dtype=torch.float32, device=dev).expand(N, OH, OW, Cout)
        if nm is None:
            nm = torch.empty(0, dtype=torch.uint8, device=dev)
        ctx.mark_non_differentiable(nm)
        ctx.set_materialize_grads(False)      # no zero-filled "gradient" for the mantissa output
        # alias: a second handle on the INPUT for the block's other branch (residual shortcut).  Its gradient then comes
        # back into THIS backward and is added inside the dgrad epilogue, instead of autograd summing two full tensors.
        xa = x.view_as(x) if alias else torch.empty(0, dtype=torch.float32, device=dev)
        return _from_mem(out), nm, xa

    @staticmethod
    def backward(ctx, g, _g_nm, g_alias):
        conv = ctx.conv
        xm, wm, k1, k2, sums, gq, bq, out, pidx = ctx.saved_tensors
        need_dx, need_dw = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        if ctx.pool is not None:
            # the pool's backward as its own launch (lbt_maxpool_bwd, 0.82 of the HBM peak), then the plain BN pass 1
            pk, ps, ppt, ppl, POH, POW = ctx.pool
            g_ = _to_mem(g)
            Np, Hp, Wp_, Cp = k2.shape        # (k1 is not saved with frozen statistics)
            gd = torch.empty(k2.shape, dtype=torch.float32, device=k2.device)
            _lib.call('lbt_maxpool_bwd', _lib.ptr(g_), _lib.ptr(pidx), Np, Hp, Wp_, Cp, pk, ps, ppt, ppl, POH, POW, _lib.ptr(gd),
                      _lib.stream(), meta=dict(bytes=gd.numel() * 4 + g_.numel() * 5))
            g = _from_mem(gd)
        if ctx.frozen:
            _, gm, dgamma, dbeta, d_add = _bn_backward_frozen(ctx.bn, _to_mem(g), k2, gq, bq, out, ctx.relu_mode, ctx.has_add,
                                                              grad_site=conv.qG, want_dx=False)   # ... dfxp:300
        else:
            _, gm, dgamma, dbeta, d_add = _bn_backward(ctx.bn, _to_mem(g), k1, k2, sums, gq, bq, out, ctx.relu_mode, ctx.has_add,
                                                       grad_site=conv.qG, want_dx=False)   # ... dfxp:300
        bd = ctx.block
        if bd is not None and not ctx.block_first:
            ctx.block = None
            if need_dx and not isinstance(gm, tuple):
                # the shortcut of a downsampling block: weight gradient only; the first unit's dgrad launch adds this branch
                _, dW, _ = _conv_backward(conv, ctx.geom, xm, ctx.xkind, wm, ctx.prep, gm, False, need_dw, False)
                bd.parked = (conv, ctx.geom, ctx.xkind, wm, ctx.prep, gm)
                N, H, W, Cin = ctx.geom[:4]
                dx = torch.empty(1, dtype=torch.float32, device=gm.device).expand(N, H, W, Cin)     # shape carrier only
                return ((_from_mem(dx),) + (dW, dgamma, dbeta, (_from_mem(d_add) if d_add is not None else None)) + (None,) * 12)
        parked = bd.take() if (bd is not None and need_dx) else None
        shortcut = None
        if parked is not None:     # g_alias is the shortcut unit's shape carrier
            if not isinstance(gm, tuple) and _block_dgrad_ok(conv, ctx.geom, ctx.prep):
                shortcut = parked
                addend = None
            else:
                addend = _shortcut_dgrad(parked)
        else:
            addend = _to_mem(g_alias) if (g_alias is not None and need_dx) else None
        ctx.block = None
        if isinstance(gm, tuple):        # 9..16-bit gradient: (hi, lo) byte planes
            dx, dW, _ = _conv_backward16(conv, ctx.geom, xm, ctx.xkind, wm, ctx.prep, gm[0], gm[1], need_dx, need_dw, False, addend=addend)
        else:
            dx, dW, _ = _conv_backward(conv, ctx.geom, xm, ctx.xkind, wm, ctx.prep, gm, need_dx, need_dw, False, addend=addend,
                                       shortcut=shortcut)
        return ((_from_mem(dx) if dx is not None else None), dW, dgamma, dbeta,
                (_from_mem(d_add) if d_add is not None else None)) + (None,) * 12


FUSE_UNITS = True     # module switch for the Conv2d_q + BatchNorm2d_q fused units (tests compare both settings); in eval mode it
                      # also selects the running-statistics kernels of a stand-alone BatchNorm2d_q (off: the eager reference path)
DUAL_WGRAD = os.environ.get('LBT_DUAL_WGRAD', '1') != '0'   # 16-bit gradients: weight gradient of both byte planes in one launch
DUAL_HALO = os.environ.get('LBT_DUAL_HALO', '1') != '0'     # 16-bit gradients: stride-1 3x3 input gradients through lbt_conv_i8_fprop_dual
FUSE_NEXT2 = os.environ.get('LBT_FUSE_NEXT2', '1') != '0'   # a strided block's shortcut convolution gets its input mantissas from the
                      # kernel that produced the block input too (lbt_bn_fwd_apply2) instead of a separate lbt_quantize


def _unit_fusable(conv, bn, x, running=False):
    return (FUSE_UNITS and isinstance(conv, Conv2d_q) and isinstance(bn, BatchNorm2d_q) and conv.bias is None and conv.fuse_bn and
            bn._can_fuse_c(conv.weight.shape[3], 4, running) and conv.qG.bits <= 16 and conv.qW.bits <= 8 and conv.qX.bits <= 9 and
            x.is_cuda)


def conv_bn_unit(conv, bn, x, add=None, relu=False, next_conv=None, want_fp32=True, alias=False, pool=None, block=None):
    """``bn(conv(x), add=add, relu=relu)`` as ONE fused unit when the shapes allow (else exactly that expression).

    next_conv: the Conv2d_q that consumes the result — its input quantiser then runs inside this unit's last kernel
    and the mantissas travel with the returned tensor (``_lbt_q``); want_fp32=False (only legal when next_conv is the
    ONLY consumer) skips the fp32 tensor altogether."""
    relu = relu or getattr(bn, 'relu', False)
    running = isinstance(bn, BatchNorm2d_q) and bn._running(x, add, conv.weight)
    frozen = isinstance(bn, BatchNorm2d_q) and not running and bn._frozen()    # frozen statistics with a backward pass
    if not _unit_fusable(conv, bn, x, running):
        y = bn(conv(x), add=add, relu=relu) if isinstance(bn, BatchNorm2d_q) else bn(conv(x))
        if pool is not None:
            y = pool(y)
        return (y, x) if alias else y
    pgeom = None
    if pool is not None:      # ``pool``: a MaxPool_q that consumes the unit's output and nothing else does
        if add is not None or alias or not pool_fusable(pool):
            y = conv_bn_unit(conv, bn, x, add=add, relu=relu, alias=alias)
            return (pool(y[0]), y[1]) if alias else pool(y)
        Hc, Wc = _conv_geom(conv, x, conv.weight)[11:13]
        pgeom = pool.geometry(Hc, Wc)
        if not FUSE_POOL_FWD:
            next_conv = None  # two kernels: the consumer quantises the POOLED tensor itself
    next_conv2 = None
    if isinstance(next_conv, (tuple, list)):      # two consumers of the result (a block's first 3x3 and its 1x1 shortcut convolution)
        next_conv, next_conv2 = (tuple(next_conv) + (None, None))[:2]

    def _site_of(nc):
        if nc is not None and isinstance(nc, Conv2d_q) and nc.fuse_bn:
            nb = nc.qX.bits
            if nb <= 8:
                return nc.qX, Q.MANT_S8
            if nb == 9 and relu and not nc.input_signed:
                return nc.qX, Q.MANT_U8
        return None, Q.MANT_NONE

    next_site, next_kind = _site_of(next_conv)
    next2 = None
    if next_site is not None and next_conv2 is not None and pool is None and FUSE_NEXT2:
        s2, k2_ = _site_of(next_conv2)
        if s2 is not None and s2 is not next_site:
            next2 = [s2, k2_, None]
    if next_site is None or add is not None or pool is not None:
        want_fp32 = True
    # measured: folding pays while the dgrad output is narrow (ResNet-18/20 blocks: -1.6 % step time); for the 256..2048-
    # channel block inputs of ResNet-50 the epilogue-bound 1x1 dgrad GEMMs lose more than the coalesced add costs (+3 %)
    # block (a downsampling block's _BlockDgrad): the shortcut's gradient joins inside the first unit's input-gradient launch,
    # so the alias pays at every width (frozen statistics keep both: that unit has a backward pass)
    block = block if (FUSE_BLOCK_DGRAD and not running) else None
    use_alias = bool(alias and x.requires_grad and not getattr(x, '_lbt_hollow', False) and
                     (conv.weight.shape[2] <= 128 or (block is not None and tuple(conv.stride) != (1, 1) and conv.qG.bits <= 8)))
    out, nm, xa = _ConvBNFn.apply(x, conv.weight, bn[1].gamma, bn[1].beta, add, conv, bn, relu, next_site, next_kind,
                                  want_fp32, use_alias, pgeom, next2, running, block, frozen)
    if next_site is not None and nm.numel():       # (empty: the pooled one-kernel path declined, the consumer quantises itself)
        out._lbt_q = {id(next_site): (nm, next_kind)}
        if next2 is not None and next2[2] is not None:
            out._lbt_q[id(next2[0])] = (next2[2], next2[1])
    if not want_fp32:
        out._lbt_hollow = True
    if alias:
        return out, (xa if use_alias else x)
    return out


def run_layers(layers, x, next_conv=None):
    """Forward through a layer list with the Conv2d_q -> BatchNorm2d_q peephole: adjacent pairs run as fused units
    and hand mantissas to the convolution that follows (``next_conv`` = the consumer after the last layer)."""
    layers = list(layers)
    i = 0
    while i < len(layers):
        m = layers[i]
        nxt = layers[i + 1] if i + 1 < len(layers) else None
        if isinstance(m, Conv2d_q) and isinstance(nxt, BatchNorm2d_q):
            after = layers[i + 2] if i + 2 < len(layers) else next_conv
            if FUSE_POOL_FWD and isinstance(after, MaxPool_q) and i + 2 < len(layers):
                after2 = layers[i + 3] if i + 3 < len(layers) else next_conv
                x = conv_bn_unit(m, nxt, x, pool=after, next_conv=_first_conv(after2))   # conv -> BN -> ReLU -> max-pool (ImageNet stem)
                i += 3
                continue
            x = conv_bn_unit(m, nxt, x, next_conv=_first_conv(after))
            i += 2
        elif isinstance(m, ResidualBlock_q):
            x = m(x, next_conv=_first_conv(nxt if nxt is not None else next_conv))
            i += 1
        else:
            x = m(x)
            i += 1
    return x


def _first_conv(m):
    """The Conv2d_q that quantises the input of module ``m`` FIRST AND ONLY ONCE per site, or None."""
    if isinstance(m, Conv2d_q):
        return m
    if isinstance(m, ResidualBlock_q):
        first = m.residual[0] if isinstance(m.residual[0], Conv2d_q) else None
        sc = list(m.shortcut) if isinstance(m.shortcut, nn.Sequential) else []
        if first is not None and sc and isinstance(sc[0], Conv2d_q):
            return (first, sc[0])          # both read the block input, each through its own quantiser
        return first
    return None


class BatchNorm2d_q(nn.Sequential):
    """dfxp:697-743: Normalization_q then Rescale_q (whose input range is hard-coded to 2, dfxp:735).

    In training mode with <= 8-bit activation quantisers, <= 16-bit gradient quantisers and C % 4 == 0 the pair runs as the fused kernels of
    csrc/bn.cu; ``forward(x, add=None, relu=False)`` can additionally fold the residual sum and the ReLU
    that follow it in the reference's blocks (dfxp:862, 986).  In eval mode the same kernels normalise with the running
    statistics (dfxp:616) when no autograd graph is recorded (see ``_running``).  ``freeze_statistics()``: training mode
    with the running statistics, which are then never updated (frozen batch-norm for quantisation-aware fine-tuning); the
    forward pass runs the eval kernels, the backward pass is ONE launch (lbt_bn_bwd_running).  Otherwise the two
    sub-modules run one after the other (Normalization_q honours ``frozen`` too)."""

    def __init__(self, bits, num_features, momentum=0.999, eps=1e-5, *, weight_decay=0.0, target_overflow_rate=0.0,
                 input_range=2, gamma_range=2, beta_range=2, grad_range=2, grad_bits=None, name='bn', runtime=None,
                 fused=True, relu=False):
        super().__init__(
            Normalization_q(bits, num_features, momentum, eps, target_overflow_rate=target_overflow_rate,
                            input_range=input_range, grad_range=grad_range, grad_bits=grad_bits, name=name + '-norm',
                            runtime=runtime),
            Rescale_q(bits, num_features, weight_decay=weight_decay, target_overflow_rate=target_overflow_rate,
                      input_range=2, gamma_range=gamma_range, beta_range=beta_range, grad_range=grad_range,
                      grad_bits=grad_bits, name=name + '-rescale', runtime=runtime))
        self.fused = fused
        self.relu = relu            # apply the ReLU that follows this BN in the reference's layer lists

    @property
    def frozen(self):
        return self[0].frozen

    def freeze_statistics(self, flag=True):
        """Frozen statistics (flag=True) or not: in training mode the layer then normalises with the running averages and
        never updates them; gamma and beta still train, and all four quantisers run as in training.  Eval mode is unaffected.
        Returns self."""
        self[0].frozen = bool(flag)
        return self

    def _frozen(self):
        """Training mode with frozen statistics."""
        return self.training and self[0].frozen

    def _can_fuse_c(self, C, dim, running=False):
        norm, resc = self[0], self[1]
        # frozen statistics with a backward pass: on the kernels only with FUSE_UNITS on (off: the eager reference path)
        return (self.fused and (running or (self.training and (FUSE_UNITS or not norm.frozen))) and dim in (2, 4) and C % 4 == 0 and
                max(norm.qX.bits, resc.qX.bits) <= 8 and max(norm.qG.bits, resc.qG.bits) <= 16 and
                min(norm.qX.bits, resc.qX.bits, norm.qG.bits, resc.qG.bits) >= 2)

    def _can_fuse(self, x, running=False):
        return self._can_fuse_c(x.shape[1], x.dim(), running)

    def _running(self, *inputs):
        """Eval mode (or frozen statistics) on the fused kernels without a backward pass: normalise with the running
        statistics.  Only where no autograd graph is recorded (eval mode with gradients keeps the eager path; frozen statistics
        with a graph take the frozen path, see ``_frozen``), and only with FUSE_UNITS on (off, the eager reference arithmetic)."""
        if (self.training and not self[0].frozen) or not FUSE_UNITS:
            return False
        return not torch.is_grad_enabled() or not any(t is not None and t.requires_grad
                                                      for t in inputs + (self[1].gamma, self[1].beta))

    def forward(self, x, add=None, relu=False):
        relu = relu or self.relu
        running = self._running(x, add)
        if self._can_fuse(x, running):
            return _FusedBNFn.apply(x, self[1].gamma, self[1].beta, add, self, relu, running, not running and self._frozen())
        y = self[1](self[0](x))
        if add is not None:
            y = y + add
        return _ReLUFn.apply(y) if relu else y

    def info(self):
        return 'BatchNorm'


BatchNorm_q = BatchNorm2d_q


# ------------------------------------------------------------------------------------------------
# Plumbing layers (dfxp:983-1053) with TF semantics
# ------------------------------------------------------------------------------------------------


class _ReLUFn(torch.autograd.Function):
    """lbt_relu: tf.maximum(0.0, X) and its gradient (to X only where X > 0)."""

    @staticmethod
    def forward(ctx, x):
        x = _mem_contig(x)
        y = torch.empty_like(x)
        _lib.call('lbt_relu', _lib.ptr(x), None, _lib.ptr(y), x.numel(), _lib.stream(), meta=dict(bytes=x.numel() * 8))
        ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, g):
        (y,) = ctx.saved_tensors
        g = _mem_contig(g)              # same memory order as y (channels_last for 4-D)
        dx = torch.empty_like(y)
        _lib.call('lbt_relu', _lib.ptr(y), _lib.ptr(g), _lib.ptr(dx), y.numel(), _lib.stream(), meta=dict(bytes=y.numel() * 12))
        return dx


class ReLU_q(nn.Module):
    """dfxp:983-990."""

    def forward(self, x):
        _require_cuda_f32(x, 'ReLU_q')
        return _ReLUFn.apply(x)

    def info(self):
        return 'ReLU'


class _MaxPoolFn(torch.autograd.Function):
    """lbt_maxpool_fwd / lbt_maxpool_bwd on the NHWC memory of a channels_last tensor."""

    @staticmethod
    def forward(ctx, x, k, s, pt, pl, OH, OW):
        x_ = _to_mem(x)
        N, H, W, C = x_.shape
        out = torch.empty(N, OH, OW, C, dtype=torch.float32, device=x.device)
        idx = torch.empty(N, OH, OW, C, dtype=torch.uint8, device=x.device)
        _lib.call('lbt_maxpool_fwd', _lib.ptr(x_), N, H, W, C, k, s, pt, pl, OH, OW, _lib.ptr(out), _lib.ptr(idx),
                  _lib.stream(), meta=dict(bytes=x_.numel() * 4 + out.numel() * 5))
        ctx.geom = (N, H, W, C, k, s, pt, pl, OH, OW)
        ctx.save_for_backward(idx)
        return _from_mem(out)

    @staticmethod
    def backward(ctx, g):
        (idx,) = ctx.saved_tensors
        N, H, W, C, k, s, pt, pl, OH, OW = ctx.geom
        g_ = _to_mem(g)
        dx = torch.empty(N, H, W, C, dtype=torch.float32, device=g.device)
        _lib.call('lbt_maxpool_bwd', _lib.ptr(g_), _lib.ptr(idx), N, H, W, C, k, s, pt, pl, OH, OW, _lib.ptr(dx),
                  _lib.stream(), meta=dict(bytes=g_.numel() * 5 + dx.numel() * 4))
        return _from_mem(dx), None, None, None, None, None, None


class MaxPool_q(nn.Module):
    """tf.nn.max_pool with 'SAME' (padding ignored in the max) or 'VALID' (dfxp:993-1006)."""

    def __init__(self, kernel_size, stride, padding='SAME'):
        super().__init__()
        self.k, self.s, self.padding = kernel_size, stride, padding

    def geometry(self, H, W):
        """(k, s, pad_top, pad_left, OH, OW) on an H x W grid."""
        if self.padding == 'SAME':
            OH, pt, pb = same_pad(H, self.k, self.s)
            OW, pl, pr = same_pad(W, self.k, self.s)
        else:
            pt = pl = 0
            OH, OW = (H - self.k) // self.s + 1, (W - self.k) // self.s + 1
        return self.k, self.s, pt, pl, OH, OW

    def forward(self, x):
        H, W = x.shape[2], x.shape[3]
        _, _, pt, pl, OH, OW = self.geometry(H, W)
        _require_cuda_f32(x, 'MaxPool_q')
        if x.dim() != 4 or self.k > 15:
            raise _lib.LbtError('MaxPool_q: needs a 4-d tensor and a window of at most 15x15')
        return _MaxPoolFn.apply(x, self.k, self.s, pt, pl, OH, OW)


def pool_fusable(pool):
    """A MaxPool_q that conv_bn_unit takes into the fused unit (``pool``): at most 2 x 2 windows over a pixel."""
    return isinstance(pool, MaxPool_q) and pool.k <= 2 * pool.s and pool.k <= 15


class _AvgPoolFn(torch.autograd.Function):
    """lbt_avgpool_fwd / lbt_avgpool_bwd on the NHWC memory of a channels_last tensor ('VALID' windows)."""

    @staticmethod
    def forward(ctx, x, k, s):
        x_ = _to_mem(x)
        N, H, W, C = x_.shape
        OH, OW = (H - k) // s + 1, (W - k) // s + 1
        out = torch.empty(N, OH, OW, C, dtype=torch.float32, device=x.device)
        _lib.call('lbt_avgpool_fwd', _lib.ptr(x_), N, H, W, C, k, s, OH, OW, _lib.ptr(out), _lib.stream(),
                  meta=dict(bytes=(x_.numel() + out.numel()) * 4))
        ctx.geom = (N, H, W, C, k, s, OH, OW)
        return _from_mem(out)

    @staticmethod
    def backward(ctx, g):
        N, H, W, C, k, s, OH, OW = ctx.geom
        g_ = _to_mem(g)
        dx = torch.empty(N, H, W, C, dtype=torch.float32, device=g.device)
        _lib.call('lbt_avgpool_bwd', _lib.ptr(g_), N, H, W, C, k, s, OH, OW, _lib.ptr(dx), _lib.stream(),
                  meta=dict(bytes=(g_.numel() + dx.numel()) * 4))
        return _from_mem(dx), None, None


class AvgPool_q(nn.Module):
    """tf.nn.avg_pool 'VALID' (dfxp:1009-1022)."""

    def __init__(self, kernel_size, stride=1):
        super().__init__()
        self.k, self.s = kernel_size, stride

    def forward(self, x):
        _require_cuda_f32(x, 'AvgPool_q')
        if x.dim() != 4:
            raise _lib.LbtError('AvgPool_q: needs a 4-d tensor')
        return _AvgPoolFn.apply(x, self.k, self.s)


class _XentFn(torch.autograd.Function):
    """Mean sparse softmax cross-entropy (models.py:30-32) and its gradient: lbt_softmax_xent_fwd / _bwd."""

    @staticmethod
    def forward(ctx, logits, labels):
        logits = logits.contiguous()
        B, C = logits.shape
        probs = torch.empty_like(logits)
        loss = torch.empty((), dtype=torch.float32, device=logits.device)
        _lib.call('lbt_softmax_xent_fwd', _lib.ptr(logits), _lib.ptr(labels), B, C, _lib.ptr(probs), _lib.ptr(loss), _lib.stream())
        ctx.save_for_backward(probs, labels)
        return loss

    @staticmethod
    def backward(ctx, gout):
        probs, labels = ctx.saved_tensors
        B, C = probs.shape
        d = torch.empty_like(probs)
        _lib.call('lbt_softmax_xent_bwd', _lib.ptr(probs), _lib.ptr(labels), _lib.ptr(gout.contiguous()), B, C, _lib.ptr(d),
                  _lib.stream())
        return d, None


def softmax_cross_entropy(logits, labels):
    """reduce_mean(sparse_softmax_cross_entropy_with_logits) of models.py:30-32."""
    _require_cuda_f32(logits, 'softmax_cross_entropy')
    if logits.dim() != 2 or not labels.is_cuda:
        raise _lib.LbtError('softmax_cross_entropy: expects [batch, classes] logits and CUDA integer labels')
    return _XentFn.apply(logits, labels.to(torch.int64).contiguous())


class _DropoutFn(torch.autograd.Function):
    """lbt_dropout: x / keep * floor(keep + u); the backward recomputes the mask from the same uniforms / Philox stream."""

    @staticmethod
    def forward(ctx, x, keep, u, seed, offset, dev_step):
        x = _mem_contig(x)
        y = torch.empty_like(x)
        _lib.call('lbt_dropout', _lib.ptr(x), _lib.ptr(u), float(keep), int(seed), int(offset), _lib.ptr(dev_step), _lib.ptr(y),
                  x.numel(), _lib.stream(), meta=dict(bytes=x.numel() * 8))
        ctx.args = (keep, seed, offset, dev_step)
        ctx.fmt4 = x.dim() == 4
        ctx.save_for_backward(u)
        return y

    @staticmethod
    def backward(ctx, g):
        (u,) = ctx.saved_tensors
        keep, seed, offset, dev_step = ctx.args
        g = _mem_contig(g)
        dx = torch.empty_like(g)
        _lib.call('lbt_dropout', _lib.ptr(g), _lib.ptr(u), float(keep), int(seed), int(offset), _lib.ptr(dev_step), _lib.ptr(dx),
                  g.numel(), _lib.stream(), meta=dict(bytes=g.numel() * 8))
        return dx, None, None, None, None, None


class Dropout_q(nn.Module):
    """tf.nn.dropout(x, keep_prob) = x / keep * floor(keep + u) (dfxp:1025-1040); keep_prob is KEEP."""

    def __init__(self, keep_prob, runtime=None):
        super().__init__()
        self.keep_prob = keep_prob
        self.uniform_fn = None      # tests: callable(x) -> the reference's uniform tensor (memory order of x)
        self.runtime = runtime or default_runtime()
        self.did = self.runtime.next_dropout_id()      # per model, not per process: a resumed run replays the same stream

    def forward(self, x):
        if not self.training or self.keep_prob >= 1.0:
            return x
        _require_cuda_f32(x, 'Dropout_q')
        rt = self.runtime
        if self.uniform_fn is not None:
            u = _mem_contig(self.uniform_fn(x).to(torch.float32))
            return _DropoutFn.apply(x, self.keep_prob, u, 0, 0, None)
        # Philox stream disjoint from the quantisers': ids count down from 2^31
        return _DropoutFn.apply(x, self.keep_prob, None, rt.seed, Q.make_offset(0x7fffffff - self.did, 0), rt.dev_step)


class Flatten_q(nn.Module):
    """tf.reshape(X, [-1, dim]) of the NHWC tensor (dfxp:1043-1053)."""

    def __init__(self, dim):
        super().__init__()
        self.dim = dim

    def forward(self, x):
        if x.dim() == 4:
            x = x.permute(0, 2, 3, 1)
        return x.reshape(-1, self.dim)


class _GradBufferFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, layer):
        ctx.layer = layer
        return x.view_as(x)

    @staticmethod
    def backward(ctx, dy):
        layer = ctx.layer
        site, rt = layer.qG, layer.qG.runtime
        g = _to_mem(dy).contiguous()                    # TF layout: [batch, ...]
        n_outer = layer.buffer.shape[0]
        n_inner = layer.buffer.numel() // n_outer
        if g.shape[0] > n_outer or g.numel() // max(1, g.shape[0]) != n_inner:
            raise _lib.LbtError('GradientBuffer_q: gradient %s does not fit the buffer %s' % (tuple(g.shape), tuple(layer.buffer.shape)))
        out = torch.empty_like(g)
        if rt.noise_fn is not None:
            mode, noise, dev_step = Q.ROUND_NOISE, rt.noise_fn(site, n_inner, g.device).contiguous(), None
        else:
            mode, noise, dev_step = Q.ROUND_PHILOX, None, rt.dev_step
        _lib.call('lbt_quantize_residual', _lib.ptr(g), g.shape[0], _lib.ptr(layer.buffer), n_outer, n_inner, site.bits,
                  _lib.ptr(site.range), mode, _lib.ptr(noise), rt.seed, Q.make_offset(site.qid, 0), _lib.ptr(dev_step),
                  _lib.ptr(out), _lib.ptr(site.counters), _lib.stream(), meta=dict(bytes=n_outer * n_inner * 16))
        return _from_mem(out), None


class GradientBuffer_q(nn.Module):
    """dfxp:473-509: error-feedback gradient quantiser.  Identity forward; backward quantises ``grad + buffer``
    (stochastic) and keeps the rounding residual in ``buffer`` for the next step (one pass: lbt_quantize_residual).
    ``shape`` is the gradient's shape in the reference's layout ([batch, H, W, C] or [batch, features]); a shorter
    last batch is zero-padded along dim 0 (dfxp:495-499) and the result sliced back (dfxp:506)."""

    def __init__(self, bits, shape, *, target_overflow_rate=0.0, grad_range=2, name='grad_buffer', runtime=None):
        super().__init__()
        rt = runtime or default_runtime()
        self.bits, self.name = bits, name
        self.register_buffer('buffer', torch.zeros(*shape))                                    # dfxp:490-491
        self.qG = QuantSite(rt, name + '/grad', bits, grad_range, target_overflow_rate)          # dfxp:492-493

    def forward(self, x):
        return _GradBufferFn.apply(x, self)

    def info(self):
        return 'Gradient buffer'


class Sequential_q(nn.Sequential):
    """dfxp:512-536."""


# ------------------------------------------------------------------------------------------------
# Residual blocks (dfxp:746-980)
# ------------------------------------------------------------------------------------------------


class ResidualBlock_q(nn.Module):
    expansion = 1

    def __init__(self, bits, in_channels, channels, stride, batch_norm=True, *, weight_decay=0.0, target_overflow_rate=0.0,
                 input_range=2, weight_range=2, bias_range=2, grad_range=2, grad_bits=None, name='block', runtime=None):
        super().__init__()
        ckw = dict(bias=not batch_norm, weight_decay=weight_decay, input_range=input_range, weight_range=weight_range,
                   bias_range=bias_range, grad_range=grad_range, grad_bits=grad_bits, input_signed=False, runtime=runtime)
        # relu=True folds the ReLU that follows the BN in the reference (dfxp:795, 928) into the BN kernels
        self._bn = lambda n, c, relu=False: (
            BatchNorm2d_q(bits, c, weight_decay=weight_decay, target_overflow_rate=target_overflow_rate,
                          input_range=input_range, grad_range=grad_range, grad_bits=grad_bits, name=n, runtime=runtime,
                          relu=relu) if batch_norm else (ReLU_q() if relu else nn.Identity()))
        self.residual = self._build_residual(bits, in_channels, channels, stride, name, ckw)
        if stride == 1 and in_channels == self.expansion * channels:                           # dfxp:828-829
            self.shortcut = nn.Sequential()
        else:
            self.shortcut = nn.Sequential(
                Conv2d_q(bits, in_channels, self.expansion * channels, 1, stride, 'SAME', name=name + '-shortcut',
                         target_overflow_rate=target_overflow_rate, **ckw),
                self._bn(name + '-shortcut-bn', self.expansion * channels))
        del self._bn

    def _build_residual(self, bits, in_channels, channels, stride, name, ckw):
        return nn.Sequential(
            Conv2d_q(bits, in_channels, channels, 3, stride, 'SAME', name=name + '-1', **ckw),
            self._bn(name + '-bn1', channels, relu=True),
            Conv2d_q(bits, channels, channels, 3, 1, 'SAME', name=name + '-2', **ckw),
            self._bn(name + '-bn2', channels))

    def forward(self, x, next_conv=None):
        # y = relu(residual(x) + shortcut(x)) (dfxp:858-863); the sum and the ReLU ride in the last BN's kernels.
        # Block inputs come from a ReLU (or a max-pool of one) in every reference model: non-negative.
        # Conv+BN pairs run as fused units (conv_bn_unit): inside the block the activations between them exist
        # only as mantissas; next_conv is the convolution that consumes the block output (wired by run_layers).
        res = list(self.residual)
        sc_layers = list(self.shortcut)
        paired = len(res) % 2 == 0 and all(isinstance(res[i], Conv2d_q) and isinstance(res[i + 1], BatchNorm2d_q)
                                           for i in range(0, len(res), 2))
        if paired:
            # the first unit hands back an alias of x for the shortcut branch: the shortcut's gradient then returns
            # through that unit's backward and is added in its dgrad epilogue (no separate add over the tensor)
            # a strided first unit and a 1x1 shortcut unit: one launch for the block's input gradient (_BlockDgrad)
            bd = _BlockDgrad() if len(sc_layers) == 2 and tuple(res[0].stride) != (1, 1) else None
            r, xs = conv_bn_unit(res[0], res[1], x, next_conv=res[2], want_fp32=False, alias=True, block=bd)
            if xs is not x and getattr(x, '_lbt_q', None) is not None:
                xs._lbt_q = x._lbt_q       # mantissas made for the shortcut convolution's quantiser travel with the alias
            for i in range(2, len(res) - 2, 2):
                r = conv_bn_unit(res[i], res[i + 1], r, next_conv=res[i + 2], want_fp32=False)
            sc = conv_bn_unit(sc_layers[0], sc_layers[1], xs, block=bd) if len(sc_layers) == 2 else self.shortcut(xs)
            return conv_bn_unit(res[-2], res[-1], r, add=sc, relu=True, next_conv=next_conv)
        r = x
        for m in res[:-1]:
            r = m(r)
        last = res[-1]
        sc = self.shortcut(x)
        if isinstance(last, BatchNorm2d_q):
            return last(r, add=sc, relu=True)
        return _ReLUFn.apply(last(r) + sc)

    def info(self):
        return 'Residual block'


class ResidualBottleneck_q(ResidualBlock_q):
    expansion = 4

    def _build_residual(self, bits, in_channels, channels, stride, name, ckw):
        return nn.Sequential(
            Conv2d_q(bits, in_channels, channels, 1, 1, 'SAME', name=name + '-1', **ckw),
            self._bn(name + '-bn1', channels, relu=True),
            Conv2d_q(bits, channels, channels, 3, stride, 'SAME', name=name + '-2', **ckw),      # stride on the 3x3
            self._bn(name + '-bn2', channels, relu=True),
            Conv2d_q(bits, channels, 4 * channels, 1, 1, 'SAME', name=name + '-3', **ckw),
            self._bn(name + '-bn3', 4 * channels))
