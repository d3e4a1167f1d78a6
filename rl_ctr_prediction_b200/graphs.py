"""CUDA-graph replay of the training step (no counterpart in the reference: its loop launches ~200 ATen kernels
per batch from Python, src/main/pretrain_main.py:96-103).

One step of LR + FM + DeepFM is ~70 kernel launches of a few tens of microseconds each; issued one by one from
Python (ctypes + autograd) the host cannot keep the GPU busy.  Every launch of the step is stream-ordered, takes its
step index from a device scalar (:class:`.tables.TableAdamState`) and allocates nothing the caching allocator cannot
serve from a private pool, so the whole step -- sort, catch-up, gather + interaction, tower GEMMs, loss, backward,
segment-reduce + Adam, dense Adam -- is captured once and replayed with new ids / labels copied into static buffers.

    step = GraphedTrainStep([(model, optimizer), ...], loss_fn)
    for features, labels in batches:            # fixed batch shape; a different shape takes the eager path
        losses = step(features, labels)         # list of device scalars, one per model

The first ``eager_steps`` calls run eagerly (they are real training steps: lazily created state -- Adam moments,
workspaces -- must exist before capture); the next call captures and replays.  Numbers are those of the eager path.
"""
from __future__ import annotations

import torch

from . import _lib
from . import p_model as Model


def eager_step(model, optimizer, loss_fn, x, y):
    """One training step of one model: the fused loss head for tower-less models, autograd for DeepFM
    (src/main/pretrain_main.py:96-102)."""
    from . import pretrain_main as PM
    if hasattr(model, "train_step"):           # sharded.ShardedCTR: the row-sharded step (device barriers, no host sync)
        return model.train_step(x, y, optimizer).detach()
    if hasattr(model, "logit") and type(loss_fn) is torch.nn.BCELoss and loss_fn.reduction == "mean" and loss_fn.weight is None:
        return fused_logit_step(model, optimizer, x, y)  # tower models: autograd for the tower, fused sigmoid + BCE head
    if getattr(model, "mlp", None) is not None:          # DeepFM, W&D, FNN, IPNN: the tower goes through autograd
        p = model(x)
        tl = loss_fn(p, y.reshape(-1, 1).float())
        model.zero_grad()
        tl.backward()
        optimizer.step()
        return tl.detach()             # keep no autograd graph alive between steps (its nodes pin a stream)
    return PM.fused_train_step(model, optimizer, x, y)


def fused_logit_step(model, optimizer, x, y):
    """The loop body of src/main/pretrain_main.py:96-102 for a model with a dense tail (DeepFM, W&D, FNN, IPNN, OPNN, DCN, AFM):
    ``model.logit(x)`` through autograd, then sigmoid + ``nn.BCELoss`` and their gradient in ONE library call
    (rlctr_bce_fwd_bwd: torch's clamped-log arithmetic, SURVEY N2) instead of torch's eight elementwise / reduction kernels,
    then ``logit.backward(dlogit)`` and the optimizer step.  Same numbers as ``loss(model(x), y); backward()``."""
    lib = _lib.load()
    z = model.logit(x)
    B = z.shape[0]
    dev = z.device
    zz = z.detach().reshape(-1).contiguous()
    yy = y.reshape(-1).contiguous()
    yi = yy if yy.dtype == torch.int64 else None
    yf = None if yi is not None else yy.float()
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    dlogit = torch.empty(B, dtype=torch.float32, device=dev)
    _lib.check(lib.rlctr_bce_fwd_bwd(_lib.ptr(zz), _lib.ptr(yi), _lib.ptr(yf), None, _lib.ptr(loss), _lib.ptr(dlogit), None,
                                     _lib.ptr(model._reduce_ws(dev)), B, _lib.stream()), "rlctr_bce_fwd_bwd")
    model.zero_grad()
    z.backward(dlogit.view_as(z))
    optimizer.step()
    return loss.reshape(())


class Prefetched:
    """A batch whose host -> device copy is in flight on the copy stream (GraphedTrainStep.prefetch)."""
    __slots__ = ("x", "y", "ready", "slot")

    def __init__(self, x, y, ready, slot):
        self.x, self.y, self.ready, self.slot = x, y, ready, slot


class GraphedTrainStep:
    def __init__(self, pairs, loss_fn=None, eager_steps=2, steps_ahead=65536, fork=True):
        self.pairs = list(pairs)
        self.loss_fn = loss_fn if loss_fn is not None else torch.nn.BCELoss()
        self.eager_left = int(eager_steps)
        self.steps_ahead = int(steps_ahead)
        self.graph = None
        self.x = self.y = None
        self.losses = None
        self.launches_per_step = 0
        self._copy_stream = None       # prefetch(): pinned host -> staging buffers, overlapped with the running step
        self._stage = [None, None]
        self._consumed = [None, None]
        self._slot = 0
        self.fork = bool(fork)         # capture tower-less models as parallel branches of the graph (see _forked)
        self._side_streams = []
        self.stream = None             # warm-up steps and the capture share one side stream (autograd's AccumulateGrad
                                       # nodes remember the stream they were created on)

    # ---- host-side bookkeeping a replay must redo (the kernels advance the device counters themselves) -----------
    def _optimizers(self):
        seen = []
        for _, opt in self.pairs:
            if opt not in seen:
                seen.append(opt)
        return seen

    def _note_replayed_step(self):
        for opt in self._optimizers():
            opt._host_step += 1
            for owner in opt._last_tables:              # the replay advanced exactly the counters the captured step did
                owner._opt.host_step += 1
                if owner._opt.lazy:
                    owner._opt.dirty = True
            opt._note_dense(opt._last_live)

    def _room(self):
        """Adam's per-step scalars are tabulated on the device; a captured graph holds the table's address, so
        the table must already cover the steps the graph will be replayed for, at the address it was captured with (an
        optimizer's load_state_dict may have grown it)."""
        if [opt._captured() for opt in self._optimizers()] != self._captured:
            return False
        for opt in self._optimizers():
            for owner in opt._tables:
                if owner._opt.host_step + 4 >= owner._opt.sched.length:
                    return False
            if float(opt.param_groups[0]["lr"]) != opt.lr:
                opt._sync_hyper()                       # re-tabulated in place: the captured graph reads the same addresses
            if opt._dense_sched is not None and opt._dense_done + 4 >= opt._dense_sched.length:
                return False
        return True

    def _reserve(self):
        for opt in self._optimizers():
            for owner in opt._tables:
                owner._opt.sched.ensure(owner._opt.host_step + self.steps_ahead)
                if owner._opt.lazy:
                    owner._opt.dirty = True     # the replays leave rows behind: the captured step must hold the catch-up (a
                                                # table just loaded or flushed is settled, and its eager step would skip it)
            if opt._dense_sched is not None:
                opt._dense_sched.ensure(opt._dense_done + self.steps_ahead)

    def _eager(self, x, y):
        return [eager_step(m, opt, self.loss_fn, x, y) for m, opt in self.pairs]

    def _branches(self):
        """Indices of the models whose step may run on a forked stream inside the capture: tower-less single-GPU models
        (their step is a handful of HBM-bound kernels: catch-up, gather, loss, segment-reduce + Adam) with an optimizer of
        their own.  They overlap the tensor-bound tower GEMMs of the models that stay on the capture stream."""
        if not self.fork:
            return []
        opts = [opt for _, opt in self.pairs]
        # a row-sharded model may branch off too when it has a process group of its own (sharded.ShardedCTR.fork_ok): its
        # collectives then run on their own communicator, so the branches' NCCL calls cannot be ordered differently on
        # different ranks, and its device barriers use the signal pads of its own symmetric allocation
        side = [i for i, (m, opt) in enumerate(self.pairs)
                if getattr(m, "mlp", None) is None and opts.count(opt) == 1 and
                ((isinstance(m, Model._TableModel) and not isinstance(m, (Model.DCN, Model.AFM))) or getattr(m, "fork_ok", False))]
        if any(hasattr(m, "train_step") and not getattr(m, "fork_ok", False) for m, _ in self.pairs):
            side = []                             # sharded models sharing one communicator: keep the step serial
        if len(side) == len(self.pairs):
            side = side[1:]                       # somebody has to stay on the capture stream
        return side

    def _forked(self, x, y):
        """The step with the tower-less models on side streams (fork after the shared sort, join before the end): the
        captured graph gets parallel branches, so the HBM-bound kernels of LR / FM run under DeepFM's GEMMs."""
        side = self._branches()
        if not side:
            return self._eager(x, y)
        main = torch.cuda.current_stream()
        first = self.pairs[side[0]][0]
        # the sorted view of the batch is shared by every model fed with it: computed before the fork
        if hasattr(first, "train_step"):
            from . import sharded as _sh
            _sh.shared_sorted_view(Model._check_ids(x), first.feature_nums, first.group)
        else:
            Model.sort_ids(Model._check_ids(x), first._geom.n_rows)
        while len(self._side_streams) < len(side):
            self._side_streams.append(torch.cuda.Stream(device=first.table.device))
        losses = [None] * len(self.pairs)
        launched = [False]

        def launch_side():
            # fork point: everything enqueued on the capture stream so far precedes the side branches
            launched[0] = True
            here = torch.cuda.current_stream()
            for k, i in enumerate(side):
                st = self._side_streams[k]
                st.wait_stream(here)
                with torch.cuda.stream(st):
                    m, opt = self.pairs[i]
                    losses[i] = eager_step(m, opt, self.loss_fn, x, y)

        # The side branches are HBM-bound; so are the first kernels of a tower model (catch-up, gather).  Fork AFTER that gather
        # (p_model._GatherInteract calls the hook once), so that the branches run beside the tower's GEMMs instead of beside
        # its gather.
        heavy = [i for i in range(len(self.pairs)) if i not in side]
        first = self.pairs[heavy[0]][0]
        if (isinstance(first, Model._TableModel) or hasattr(first, "train_step")) and getattr(first, "mlp", None) is not None:
            first._after_gather = launch_side
        else:
            launch_side()
        for i in heavy:
            m, opt = self.pairs[i]
            losses[i] = eager_step(m, opt, self.loss_fn, x, y)
        if not launched[0]:
            first._after_gather = None
            launch_side()
        for k in range(len(side)):
            main.wait_stream(self._side_streams[k])
        return losses

    def _eager_on_side_stream(self, x, y):
        if self.stream is None:
            self.stream = torch.cuda.Stream(device=self.pairs[0][0].table.device)
        cur = torch.cuda.current_stream()
        self.stream.wait_stream(cur)
        with torch.cuda.stream(self.stream):
            out = self._eager(x, y)
        cur.wait_stream(self.stream)
        return out

    def _capture(self, x, y):
        if _lib.timing():
            raise _lib.RlctrError("per-kernel timing (KernelTimer) cannot be recorded inside a graph capture")
        self._reserve()
        dev = self.pairs[0][0].table.device
        self.x = torch.empty(tuple(x.shape), dtype=x.dtype, device=dev)
        self.y = torch.empty(tuple(y.shape), dtype=y.dtype, device=dev)
        self.x.copy_(x, non_blocking=True)
        self.y.copy_(y, non_blocking=True)
        lib = _lib.load()
        torch.cuda.synchronize()
        l0 = lib.rlctr_launch_count()
        if self.stream is None:
            self.stream = torch.cuda.Stream(device=dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=self.stream):
            self.losses = self._forked(self.x, self.y)
        self.launches_per_step = int(lib.rlctr_launch_count() - l0)
        self.graph = g
        self._captured = [opt._captured() for opt in self._optimizers()]
        # the capture ran the Python side of one step (host counters advanced) but no kernel: replay it now
        g.replay()

    def prefetch(self, x, y):
        """Start copying a (pinned) host batch to the device on a side stream and return a handle ``step(handle)``
        consumes.  Call it for batch i+1 before ``step`` of batch i: the copy overlaps the running step."""
        dev = self.pairs[0][0].table.device
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=dev)
        slot = self._slot
        self._slot ^= 1
        st = self._stage[slot]
        if st is None or tuple(st[0].shape) != tuple(x.shape) or tuple(st[1].shape) != tuple(y.shape):
            st = (torch.empty(tuple(x.shape), dtype=x.dtype, device=dev), torch.empty(tuple(y.shape), dtype=y.dtype, device=dev))
            self._stage[slot] = st
            self._copy_stream.wait_stream(torch.cuda.current_stream(dev))
        cs = self._copy_stream
        if self._consumed[slot] is not None:
            cs.wait_event(self._consumed[slot])            # the step that last read this slot has taken its copy
        with torch.cuda.stream(cs):
            st[0].copy_(x, non_blocking=True)
            st[1].copy_(y, non_blocking=True)
            ready = torch.cuda.Event()
            ready.record(cs)
        return Prefetched(st[0], st[1], ready, slot)

    def losses_to_host(self, losses):
        """Start the device -> host copy of a step's losses into a pinned buffer and return ``fetch``: calling it waits
        for THAT copy only and returns the list of floats.  Fetch step i-1 after launching step i and the host never
        stalls the GPU (the reference's loop stalls it once per batch with ``train_loss.item()``)."""
        flat = torch.cat([l.reshape(-1) for l in losses])   # a co-located group returns one loss per member
        if getattr(self, "_host_losses", None) is None or self._host_losses[0].numel() != flat.numel():
            self._host_losses = [torch.empty(flat.numel(), dtype=torch.float32).pin_memory() for _ in range(3)]
            self._host_slot = 0
        buf = self._host_losses[self._host_slot]
        self._host_slot = (self._host_slot + 1) % 3
        buf.copy_(flat, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())

        def fetch():
            ev.synchronize()
            return buf.tolist()
        return fetch

    def __call__(self, x, y=None):
        if isinstance(x, Prefetched):
            h = x
            torch.cuda.current_stream().wait_event(h.ready)
            out = self._run(h.x, h.y)
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream())
            self._consumed[h.slot] = ev
            return out
        return self._run(x, y)

    def _run(self, x, y):
        dev = self.pairs[0][0].table.device
        if self.graph is not None and tuple(x.shape) == tuple(self.x.shape) and self._room():
            self.x.copy_(x, non_blocking=True)
            self.y.copy_(y, non_blocking=True)
            self.graph.replay()
            self._note_replayed_step()
            return self.losses
        if self.graph is not None and tuple(x.shape) == tuple(self.x.shape):
            self.graph = None                      # schedule table exhausted: it will be re-tabulated and re-captured
        if self.graph is None and self.eager_left <= 0 and (self.x is None or tuple(x.shape) == tuple(self.x.shape)):
            self._capture(x, y)
            return self.losses
        # warm-up steps, and batches of another shape (the last partial batch of an epoch): the eager path
        if self.graph is None:
            self.eager_left -= 1
        return self._eager_on_side_stream(x.to(dev, non_blocking=True), y.to(dev, non_blocking=True))


class GraphedCallable:
    """CUDA-graph replay of any device-only step ``fn(*tensors) -> tensor | tuple of tensors`` whose optimizers are
    :class:`.optim.Adam` (the REINFORCE step of PG_model.PolicyGradient.fused_step, an inference pass ...): the first
    ``eager_steps`` calls run eagerly on a side stream (lazily created state must exist before capture), the next one is
    captured, later ones copy the inputs into the static buffers and replay.  ``fn`` must not synchronise with the host."""

    def __init__(self, fn, optimizers=(), eager_steps=2, steps_ahead=65536):
        self.fn, self.optimizers = fn, list(optimizers)
        self.eager_left, self.steps_ahead = int(eager_steps), int(steps_ahead)
        self.graph, self.inputs, self.outputs, self.stream = None, None, None, None
        self.launches_per_step = 0

    def _note(self):
        for opt in self.optimizers:
            opt._host_step += 1
            for owner in opt._last_tables:
                owner._opt.host_step += 1
                if owner._opt.lazy:
                    owner._opt.dirty = True
            opt._note_dense(opt._last_live)

    def _reserve(self):
        for opt in self.optimizers:
            for owner in opt._tables:
                owner._opt.sched.ensure(owner._opt.host_step + self.steps_ahead)
                if owner._opt.lazy:
                    owner._opt.dirty = True     # the captured step must hold the catch-up (GraphedTrainStep._reserve)
            if opt._dense_sched is not None:
                opt._dense_sched.ensure(opt._dense_done + self.steps_ahead)

    def __call__(self, *tensors):
        dev = tensors[0].device
        if self.stream is None:
            self.stream = torch.cuda.Stream(device=dev)
        if self.graph is not None and [opt._captured() for opt in self.optimizers] != self._captured:
            self.graph = None              # an optimizer's load_state_dict replaced a tensor the graph reads: capture again
        if self.graph is not None:
            for buf, t in zip(self.inputs, tensors):
                buf.copy_(t, non_blocking=True)
            self.graph.replay()
            self._note()
            return self.outputs
        if self.eager_left > 0:
            self.eager_left -= 1
            cur = torch.cuda.current_stream()
            self.stream.wait_stream(cur)
            with torch.cuda.stream(self.stream):
                out = self.fn(*tensors)
            cur.wait_stream(self.stream)
            return out
        if _lib.timing():
            raise _lib.RlctrError("per-kernel timing (KernelTimer) cannot be recorded inside a graph capture")
        self._reserve()
        self.inputs = [torch.empty_like(t) for t in tensors]
        for buf, t in zip(self.inputs, tensors):
            buf.copy_(t, non_blocking=True)
        lib = _lib.load()
        torch.cuda.synchronize()
        l0 = lib.rlctr_launch_count()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=self.stream):
            self.outputs = self.fn(*self.inputs)
        self.launches_per_step = int(lib.rlctr_launch_count() - l0)
        self.graph = g
        self._captured = [opt._captured() for opt in self.optimizers]
        g.replay()                      # the capture ran the host side of one step but no kernel: replay it now
        return self.outputs
