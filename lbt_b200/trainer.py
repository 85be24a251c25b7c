"""The training step of the DFXP path (``trainer.py:N`` = /root/reference/trainer.py:N).

One ``Trainer.step(X, y)`` is one ``sess.run([train_op, update_range_op])`` (trainer.py:157-160):
forward, loss, backward (the layers quantise their own gradients), momentum SGD on the fp32 master
weights (trainer.py:79-84), then the range controller of every quantiser.  New here (the reference
is single-device, SURVEY.md F11): data parallelism over the batch — one process per GPU, the
gradients reduced over the replicas and the overflow counters summed before the controller runs, so
every replica keeps identical ranges and sees the global-batch overflow rate.  On GPUs the whole
exchange is ONE kernel over NVLink peer memory (lbt_dp_step: reduce-scatter by peer loads, momentum
SGD on the owned slice, all-gather of the updated weights by peer stores, counter sum + controller);
``dp='nccl'`` keeps the two-all-reduce formulation (also what the gloo CPU tests drive).

Per step the parameter side costs four launches regardless of depth: lbt_param_prep (quantise + pack
every parameter), lbt_finalize_multi (every gradient), lbt_sgd_momentum, lbt_update_ranges.
"""
import os
import sys

import torch
import torch.distributed as dist

from . import _lib
from .dfxp import ParamPrep


def sync_replicas(flat_g, counters, group=None, sync_counters=True):
    """The data-parallel exchange (SURVEY §8e): sum the flat gradient and the quantisers' overflow counters over
    the replicas.  Device-agnostic (NCCL on GPUs; the gloo CPU tests drive it too)."""
    dist.all_reduce(flat_g, op=dist.ReduceOp.SUM, group=group)
    if sync_counters:
        dist.all_reduce(counters, op=dist.ReduceOp.SUM, group=group)


class GradSink:
    """Collects (integer sum, scale exponents, weight-decay term) of every parameter gradient during backward and
    converts them all with ONE lbt_finalize_multi launch, writing straight into the flat gradient buffer."""

    def __init__(self, params):
        self.out = {id(p): p for p in params}
        self.jobs = []
        self._key = {}               # per launch slot ('all' | 'head' | 'tail'): the uploaded job table and what it describes
        self._table = {}
        self._head = 0               # jobs already finalised by flush_head()
        self._pinned = []            # staging copies of uploaded tables (kept alive for captured CUDA graphs)
        self.active = False         # only between begin() and flush(): outside a Trainer step layers finalise themselves

    def accepts(self, param):
        return self.active and id(param) in self.out

    def begin(self):
        self.jobs = []
        self._head = 0
        self.active = True

    def add(self, param, acc, ibA, ibB, exp_const, add_scale):
        self.jobs.append((param, acc, ibA, ibB, int(exp_const), float(add_scale)))

    def _launch(self, jobs, slot):
        structs, key, start = [], [], 0
        for param, acc, ibA, ibB, e, s in jobs:
            n = acc.numel()
            assert n == param.numel() and acc.is_contiguous()
            j = _lib.FinalizeJob(acc64=acc.data_ptr(), n=n, ibA=_lib.ptr(ibA) or 0, ibB=_lib.ptr(ibB) or 0, exp_const=e,
                                 add_scale=s, add=param.data.data_ptr() if s else 0, out=param.grad.data_ptr(), start=start)
            structs.append(j)
            key.append((j.acc64, n, j.ibA, j.ibB, e, s, j.add, j.out))
            start += n
        key = tuple(key)
        if key != self._key.get(slot):            # pointers are stable from step to step: upload the table once
            self._table[slot] = _lib.to_device_table(structs, jobs[0][1].device, keep=self._pinned)
            self._key[slot] = key
        _lib.call('lbt_finalize_multi', _lib.ptr(self._table[slot]), len(structs), start, _lib.stream())

    def flush_head(self):
        """Finalise what has been collected so far on the CURRENT stream (its producers must be ordered before it): the
        first layer's backward calls this so that every other gradient is converted while its own weight-gradient kernel
        — the last one of the step, with nothing else left to overlap — is still running."""
        if not self.active or len(self.jobs) == self._head:
            return
        self._launch(self.jobs[self._head:], 'head')
        self._head = len(self.jobs)

    def flush(self):
        self.active = False
        if len(self.jobs) > self._head:
            self._launch(self.jobs[self._head:], 'tail' if self._head else 'all')


class Trainer:
    def __init__(self, model, lr=1e-2, momentum=0.9, *, process_group=None, sync_counters=True, batched=True, dp=None):
        self.model = model
        self.lr, self.momentum = float(lr), float(momentum)
        self.group = process_group
        self.world = dist.get_world_size(process_group) if (dist.is_available() and dist.is_initialized()) else 1
        self.sync_counters = sync_counters
        params = [p for p in model.parameters() if p.requires_grad]
        if not params or not params[0].is_cuda:
            raise _lib.LbtError('Trainer needs the model on a CUDA device (no CPU fallback)')
        dev = params[0].device
        self.device = dev
        rt = model.runtime
        # flatten parameters / gradients / momentum: one SGD launch and one exchange per step
        sizes = [p.numel() for p in params]
        offs, total = [], 0
        for n in sizes:
            offs.append(total)
            total += -(-n // 4) * 4                      # keep every view 16-byte aligned
        # end of the step: 'fused' = ONE lbt_dp_step launch (over peer-mapped arenas when world > 1),
        # 'nccl' = all-reduces + lbt_sgd_momentum + lbt_update_ranges + lbt_step_advance
        dp = dp or os.environ.get('LBT_DP', 'fused')
        self.dp = None
        if dp == 'fused' and (sync_counters or self.world == 1):
            from .dp import DpExchange
            ok, why = 1.0, ''
            try:
                self.dp = DpExchange(len(rt.sites), total, dev, process_group)
            except Exception as e:               # e.g. no peer access between the devices: say so, use NCCL
                if self.world == 1:
                    raise
                ok, why = 0.0, str(e)
            if self.world > 1:                   # all replicas must agree on the path; doubles as the start barrier
                torch.cuda.synchronize(dev)
                flag = torch.full((1,), ok, device=dev)
                dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=process_group)
                if not bool(flag.item()):
                    print('lbt_b200: fused data-parallel exchange unavailable (%s); using NCCL all-reduce' % (why or 'a peer failed'),
                          file=sys.stderr)
                    if self.dp is not None:
                        self.dp.close()
                    self.dp = None
        self.dp_mode = 'fused' if self.dp is not None else ('nccl' if self.world > 1 else 'unfused')
        if self.dp is not None:
            rt.finalize(dev, counters=self.dp.arena.counters)
            self.flat_w, self.flat_g = self.dp.arena.flat_w, self.dp.arena.flat_g
        else:
            rt.finalize(dev)
            self.flat_w = torch.zeros(total, dtype=torch.float32, device=dev)
            self.flat_g = torch.zeros(total, dtype=torch.float32, device=dev)
        self.flat_a = torch.zeros(total, dtype=torch.float32, device=dev)        # optimizer slots start at 0 (trainer.py:83)
        for p, o, n in zip(params, offs, sizes):
            self.flat_w[o:o + n].copy_(p.data.reshape(-1))
            p.data = self.flat_w[o:o + n].view(p.shape)
            p.grad = self.flat_g[o:o + n].view(p.shape)
        self.params = params
        self.dev_lr = torch.tensor(self.lr, dtype=torch.float32, device=dev)
        if self.world > 1:                               # replicas start from rank 0's weights
            dist.broadcast(self.flat_w, src=0, group=self.group)
        # batched parameter-side launches (identical arithmetic; batched=False keeps the per-layer launches)
        self.batched = batched
        self.sink = GradSink(params) if batched else None
        rt.grad_sink = self.sink
        rt.prep = ParamPrep(model, rt, dev) if batched else None

    def set_lr(self, lr, reset_momentum=True):
        """LR change; the reference re-creates the optimizer, zeroing momentum (trainer.py:79-84, 118-132)."""
        self.lr = float(lr)
        self.dev_lr.fill_(self.lr)
        if reset_momentum:
            self.flat_a.zero_()

    def forward_backward(self, X, y):
        rt = self.model.runtime
        self.flat_g.zero_()
        if self.batched:
            rt.begin_step(self.device)
            self.sink.begin()
        logits = self.model(X)
        loss = self.model.loss(logits, y)
        loss.backward()
        rt.join_side()                       # weight-gradient kernels run on a side stream beside the backward chain
        if self.batched:
            self.sink.flush()
        return loss.detach(), logits.detach()

    def apply(self):
        rt = self.model.runtime
        if self.dp is not None:              # the whole exchange + optimizer + controller: one kernel over NVLink
            self.dp.step(self.flat_a, self.lr, self.dev_lr, self.momentum, rt)
            rt.close_step()
            return
        if self.world > 1:
            sync_replicas(self.flat_g, rt.flat['counters'], self.group, self.sync_counters)
        _lib.call('lbt_sgd_momentum', _lib.ptr(self.flat_w), _lib.ptr(self.flat_a), _lib.ptr(self.flat_g),
                  self.flat_w.numel(), self.lr, _lib.ptr(self.dev_lr), self.momentum, 1.0 / self.world, _lib.stream())
        rt.update_ranges()

    def step(self, X, y):
        """X: [N, C, H, W] (channels_last) on the device, y: int64 labels.  Returns the loss tensor."""
        loss, _ = self.forward_backward(X, y)
        self.apply()
        return loss

    # ---- the hot loop as ONE graph launch per step (trainer.py:144-162) ------------------------------------------------
    def capture(self, X_static, y_static, warmup=2):
        """Capture ``step(X_static, y_static)`` — forward, loss, backward, exchange, optimizer, controller: ~150 launches
        on two streams — into a CUDA graph.  Afterwards ``step_graph()`` replays it on whatever ``X_static`` / ``y_static``
        hold at that moment and returns the (static) loss tensor; ``feeder()`` wraps it for pinned host batches.  All state
        a step reads or writes (weights, ranges, counters, momentum, step counter = noise position) lives on the device, so
        a replayed step is bit-identical to an eager one (tests/test_data_gpu.py).  ``warmup`` eager steps run first on a
        side stream (allocator warm-up, lazy tables); they are REAL training steps."""
        if not X_static.is_cuda or not y_static.is_cuda:
            raise _lib.LbtError('Trainer.capture needs static CUDA input tensors')
        self._static = (X_static, y_static)
        s = torch.cuda.Stream(device=self.device)
        s.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(s):
            for _ in range(int(warmup)):
                self.step(X_static, y_static)
        torch.cuda.current_stream(self.device).wait_stream(s)
        torch.cuda.synchronize(self.device)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            loss = self.step(X_static, y_static)
        torch.cuda.synchronize(self.device)
        self._graph, self._graph_loss = graph, loss
        from .dfxp import Normalization_q
        self._graph_norms = [m for m in self.model.modules() if isinstance(m, Normalization_q)]
        self._graph_frozen = [m.frozen for m in self._graph_norms]
        return self

    def _bn_mode_changed(self):
        """True when a batch-norm was frozen or unfrozen since the step was captured."""
        return any(m.frozen != f for m, f in zip(self._graph_norms, self._graph_frozen))

    def freeze_bn_statistics(self, flag=True):
        """``model.freeze_bn_statistics(flag)``; a captured step recorded in the other mode is dropped (the next ``capture``
        records the new one).  Returns self."""
        self.model.freeze_bn_statistics(flag)
        if self.captured and self._bn_mode_changed():
            self._graph = self._graph_loss = None
        return self

    @property
    def captured(self):
        return getattr(self, '_graph', None) is not None

    def step_graph(self):
        """One training step = one graph launch, on the current contents of the static inputs.  Returns the loss tensor
        (static: read it, or copy it, before the next replay overwrites it).  A step captured before the batch-norm
        statistics were frozen or unfrozen on the model raises: the graph replays the kernels of the mode it was captured in."""
        if not self.captured:
            raise _lib.LbtError('Trainer.step_graph: no step is captured (never captured, or dropped by '
                                'Trainer.freeze_bn_statistics); call capture(X_static, y_static) first')
        if self._bn_mode_changed():
            raise _lib.LbtError('Trainer.step_graph: the batch-norm statistics were frozen or unfrozen on the model after '
                                'capture(); use Trainer.freeze_bn_statistics, which drops the graph, and capture again')
        self._graph.replay()
        return self._graph_loss

    def feeder(self):
        """HostFeeder over the captured step: per-step H2D of pinned host batches on a copy stream, per-step D2H of the loss
        read one step later — the device-side replacement of the reference's feed_dict round trip (trainer.py:146-160)."""
        if not self.captured:
            raise _lib.LbtError('Trainer.feeder: call capture(X_static, y_static) first')
        return HostFeeder(self.step_graph, *self._static)

    def check(self):
        """Raise if a device-side watchdog fired: a cross-replica wait of lbt_dp_step timed out (the kernel then skips the
        optimizer and every later step: the error word is sticky).  Synchronises when data-parallel; fit() calls it once per
        epoch, state_dict() always."""
        if self.dp is not None:
            e = self.dp.error()
            if e:
                raise _lib.LbtError('lbt_dp_step: a cross-replica wait timed out (flag slot %d); the replicas are no longer '
                                    'in step — this run cannot continue' % (e - 1))

    # ---- evaluation (trainer.py:164-187) ---------------------------------------------------------------------------
    @torch.no_grad()
    def evaluate(self, X, y, batch_size=1000, running_stats=False):
        """Mean loss and accuracy over (X, y) in batches of ``batch_size`` — the reference's test loop.  Like the
        reference (its ``set_testing`` call is commented out, trainer.py:164-165, "TODO BatchNorm bug") the forward pass
        runs in TRAINING mode by default: batch statistics, stochastic quantisers; nothing is updated — no range controller
        (``update_range_op`` is not fetched), no running statistics, no step counter.
        ``running_stats=True``: the batches run in eval mode instead (``model.eval()``: batch-norm with the running
        statistics, no dropout) on the fused kernels; the module's previous mode is restored afterwards.  Quantisers stay
        stochastic, with the same per-batch noise positions, and nothing is updated either."""
        from .dfxp import Normalization_q
        rt = self.model.runtime
        norms = [] if running_stats else [m for m in self.model.modules() if isinstance(m, Normalization_q)]
        saved = [m.momentum for m in norms]
        for m in norms:
            m.momentum = 1.0                       # running <- 1.0 * running + 0.0 * batch: unchanged
        modes = [(m, m.training) for m in self.model.modules()]
        counters = rt.flat['counters'].clone()
        # the reference draws fresh quantiser / dropout noise at every sess.run (dfxp:36): every test batch gets its own
        # position of the Philox stream, disjoint from the training steps' (bit 31 of the step word), and the training
        # position is restored afterwards
        step_saved = rt.dev_step.clone()
        base = (int(step_saved.item()) & 0x7FFFF) << 12
        loss_sum, acc_sum, n_batches = 0.0, 0.0, 0
        try:
            if running_stats:
                self.model.eval()
            for i in range(0, X.shape[0], batch_size):
                xb, yb = X[i:i + batch_size], y[i:i + batch_size]
                rt.dev_step.fill_(0x80000000 | ((base + n_batches) & 0x7FFFFFFF))
                logits = self.model(xb)
                loss_sum += float(self.model.loss(logits, yb))
                acc_sum += float((logits.argmax(dim=1) == yb).float().mean())
                n_batches += 1
        finally:
            for m, mom in zip(norms, saved):
                m.momentum = mom
            for m, mode in modes:
                m.training = mode
            rt.flat['counters'].copy_(counters)    # the overflow statistics of a test batch never reach the controller
            rt.dev_step.copy_(step_saved)
        return loss_sum / max(1, n_batches), acc_sum / max(1, n_batches)          # mean of per-batch means, as trainer.py:185-186

    # ---- the epoch loop (trainer.py:109-187) ---------------------------------------------------------------------------
    def fit(self, pipeline, n_epoch, batch_size, *, lr_decay_factor=0.1, decay_epochs=(80, 120, 140), test=None, log=None,
            max_batches=None, graph=False, eval_running_stats=False, freeze_bn_epoch=None):
        """``pipeline``: lbt_b200.data.Pipeline over the device-resident training set (shuffle + flip / pad-4 / crop on
        the GPU).  The learning rate is multiplied by ``lr_decay_factor`` at epochs 80, 120 and 140 and the optimizer is
        re-created (momentum slots zeroed) exactly there (trainer.py:117-132).  ``test`` = (X, y) evaluated after each
        epoch (``eval_running_stats``: see ``evaluate(running_stats=...)``).  ``graph=True``: full batches run as replays of the captured step (capture() on first use; the pipeline
        writes each batch straight into the static inputs), a short last batch runs eagerly.  With several replicas the
        pipeline must be rank-aware (lbt_b200.data.Pipeline shards every global batch by rank).
        ``freeze_bn_epoch``: the batch-norm statistics are frozen from the start of that (0-based) epoch on and unfrozen
        before it (``freeze_bn_statistics``; a captured step is re-captured in the new mode).  The schedule is a function of
        the epoch, so a resumed run re-derives it.  None: the model's setting is left as it is.
        Returns [(epoch, last_train_loss, test_loss, test_acc)]."""
        history = []
        if self.world > 1 and getattr(pipeline, 'world', 1) != self.world:
            raise _lib.LbtError('Trainer.fit: %d replicas but the pipeline is sharded %d ways — every replica would train on '
                                'the same samples' % (self.world, getattr(pipeline, 'world', 1)))
        for epoch in range(n_epoch):
            if epoch in decay_epochs:
                self.set_lr(self.lr * lr_decay_factor, reset_momentum=True)
            if freeze_bn_epoch is not None:
                self.freeze_bn_statistics(epoch >= freeze_bn_epoch)
            loss = None
            for b, (X, y) in enumerate(pipeline.epoch(batch_size, epoch)):
                if max_batches is not None and b >= max_batches:
                    break
                if graph and X.shape[0] == batch_size:
                    if not self.captured:
                        Xs = torch.empty_like(X, memory_format=torch.channels_last) if X.dim() == 4 else torch.empty_like(X)
                        self.capture(Xs.copy_(X), torch.empty_like(y).copy_(y), warmup=0)
                    self._static[0].copy_(X)
                    self._static[1].copy_(y)
                    loss = self.step_graph().clone()
                else:
                    loss = self.step(X, y)
                if log is not None and (b + 1) % 100 == 0:
                    log('Batch %d loss %f' % (b + 1, float(loss)))
            self.check()
            tl, ta = self.evaluate(*test, running_stats=eval_running_stats) if test is not None else (None, None)
            history.append((epoch, float(loss) if loss is not None else None, tl, ta))
            if log is not None and ta is not None:
                log('Epoch %d test accuracy %f' % (epoch + 1, ta))
        return history

    # ---- checkpoint / resume (trainer.py:189-192: tf.train.Saver over all variables) -----------------------------------
    def state_dict(self):
        """Everything the reference's Saver holds — weights, every ``*_range`` variable, the BN running statistics, the
        optimizer slots — plus what the TF session held implicitly (step counter = noise stream position, lr)."""
        rt = self.model.runtime
        self.check()
        accum = self.flat_a.clone()
        if self.dp is not None and self.world > 1:       # sharded optimizer: every replica holds only its slice
            dist.all_reduce(accum, op=dist.ReduceOp.SUM, group=self.group)
        return {'model': {k: v.detach().clone() for k, v in self.model.state_dict().items()},
                'momentum_slots': accum, 'lr': self.lr, 'momentum': self.momentum,
                'step': int(rt.dev_step.item()), 'seed': rt.seed}

    def load_state_dict(self, sd):
        rt = self.model.runtime
        self.model.load_state_dict(sd['model'])            # copies into the flat views (weights, ranges, counters)
        if int(sd['seed']) != rt.seed:
            raise _lib.LbtError('checkpoint was written with noise seed %d; build the model with seed=%d to resume its stream'
                                % (sd['seed'], sd['seed']))
        self.flat_a.copy_(sd['momentum_slots'].to(self.device))
        if self.dp is not None and self.world > 1:       # keep only the slice this replica owns (see state_dict)
            lo, hi = self.dp.owned()
            self.flat_a[:lo].zero_()
            self.flat_a[hi:].zero_()
        self.lr, self.momentum = float(sd['lr']), float(sd['momentum'])
        self.dev_lr.fill_(self.lr)
        rt.dev_step.fill_(int(sd['step']))
        rt.close_step()

    def save(self, path):
        torch.save(self.state_dict(), path)

    def load(self, path):
        self.load_state_dict(torch.load(path, map_location=self.device))


class HostFeeder:
    """Feeds a (CUDA-graph captured) training step from pinned host batches without stalling the GPU — the device-side
    replacement of the reference's ``feed_dict`` round trip (trainer.py:143-160), where every step waits for its inputs to
    cross PCIe and for its loss to come back.

    The next batch is copied host -> device on a copy stream into one of two staging buffers while the current step runs;
    at step start a device-to-device copy moves it into the step's static input tensors.  Each step's loss is copied back to
    pinned host memory asynchronously and read one step later, so every step still does its own H2D input copy and its own
    D2H loss read, but neither sits on the critical path.

        feeder = HostFeeder(run_step, X_static, y_static)     # run_step() -> loss tensor (e.g. graph.replay + static loss)
        feeder.prefetch(hX0, hy0)
        for i in range(n):
            if i + 1 < n: feeder.prefetch(hX[i + 1], hy[i + 1])
            prev_loss = feeder.step()                           # python float of step i-1 (None for i == 0)
        last_loss = feeder.drain()
    """

    def __init__(self, run_step, X_static, y_static):
        self.run_step, self.Xs, self.ys = run_step, X_static, y_static
        dev = X_static.device
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.stage = [(torch.empty_like(X_static), torch.empty_like(y_static)) for _ in range(2)]
        self.ready = [torch.cuda.Event() for _ in range(2)]
        self.consumed = [torch.cuda.Event() for _ in range(2)]
        self.loss_host = [torch.zeros(1, dtype=torch.float32).pin_memory() for _ in range(2)]
        self.loss_done = [torch.cuda.Event() for _ in range(2)]
        self.fill, self.take, self.pending = 0, 0, None
        cur = torch.cuda.current_stream(dev)
        for e in self.consumed:
            e.record(cur)

    def prefetch(self, hX, hy):
        """Start the host -> device copy of the NEXT batch (pinned tensors shaped like the static inputs)."""
        s = self.fill
        self.fill ^= 1
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self.consumed[s])          # the step that last used this buffer has taken its data
            self.stage[s][0].copy_(hX, non_blocking=True)
            self.stage[s][1].copy_(hy, non_blocking=True)
            self.ready[s].record(self.copy_stream)

    def step(self):
        """Run one step on the oldest prefetched batch; returns the PREVIOUS step's loss (float) or None."""
        s = self.take
        self.take ^= 1
        cur = torch.cuda.current_stream(self.Xs.device)
        cur.wait_event(self.ready[s])
        self.Xs.copy_(self.stage[s][0], non_blocking=True)         # device to device, a few microseconds
        self.ys.copy_(self.stage[s][1], non_blocking=True)
        self.consumed[s].record(cur)
        loss = self.run_step()
        self.loss_host[s].copy_(loss.detach().reshape(1), non_blocking=True)
        self.loss_done[s].record(cur)
        prev = self.drain()
        self.pending = s
        return prev

    def drain(self):
        """Wait for and return the loss of the last step issued (None if there is none outstanding)."""
        if self.pending is None:
            return None
        s, self.pending = self.pending, None
        self.loss_done[s].synchronize()
        return float(self.loss_host[s])
