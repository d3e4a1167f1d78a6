"""``Adam`` with the constructor / ``step()`` / ``zero_grad()`` surface of ``torch.optim.Adam`` as the
reference builds it (``torch.optim.Adam(params=model.parameters(), lr=..., weight_decay=...)``,
src/main/pretrain_main.py:181), so the reference's ``train(model, optimizer, ...)`` drives it unchanged.

Embedding tables (parameters created by :mod:`.p_model`) never see a dense ``[N, D]`` gradient: the
backward pass leaves (sorted ids, dlogit, saved sums) on the module and ``step()`` runs the
deterministic sort / segment-reduce / fused Adam kernel (rlctr_rows_adam).  Every other parameter
(bias, tower, policy nets) takes the fused dense Adam kernel (rlctr_dense_adam).  Numerics are
torch's ``_single_tensor_adam`` (L2 folded into the gradient) element by element.

``mode``: 'lazy' (default; reference numbers, O(touched rows) traffic), 'dense' (the literal
reference work: every row every step), 'sparse' (untouched rows frozen -- NOT the reference).

``Adagrad`` is ``torch.optim.Adagrad`` over the same tables, records and kernels (the row kernels take the per-record step
as a policy); both share :class:`_RowOptimizer`, the step loop that :mod:`.graphs` replays.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from .tables import AdagradSchedule, AdamSchedule, TableAdagradState, TableAdamState, table_struct


class _RowOptimizer:
    """The step loop shared by :class:`Adam` and :class:`Adagrad`: embedding tables (parameters created by :mod:`.p_model`,
    :mod:`.colocated`, :mod:`.sharded`) get a table state (:mod:`.tables`) that owns the catch-up, row-update and flush
    launches; every other parameter is a replicated dense tensor updated by one multi-tensor launch per step.  A subclass
    provides ``_FIXED`` (hyper-parameters fixed after construction), ``_table_state``, ``_dense_schedule``, ``_dense_new``
    and ``_dense_launch``."""

    _FIXED = ()

    def _setup(self, params, mode, defaults):
        if not params:
            raise ValueError("optimizer got an empty parameter list")
        self.mode = mode
        self.param_groups = [dict(params=params, **defaults)]
        self._tables, self._dense = [], []
        for p in params:
            owner = getattr(p, "_rlctr_owner", None)
            if owner is not None:
                if not p.is_cuda:
                    raise _lib.RlctrError("move the model to the CUDA device before building the optimizer")
                # a fresh optimizer == fresh optimizer state (the reference re-creates its optimizer every epoch,
                # src/main/pretrain_main.py:175-181): settle what the previous one still owes first
                owner.flush()
                owner._opt = self._table_state(p.data, owner._geom)
                owner._opt.host_step = 0
                self._tables.append(owner)
            else:
                self._dense.append(p)
        self._dense_state = {}
        self._dense_index = {p: i for i, p in enumerate(self._dense)}
        self._dense_count = [0] * len(self._dense)      # host mirror of the per-parameter device step counters
        self._dense_steps = None                        # int32 [len(dense)] on the device
        self._dense_sched = None
        self._last_live = []                            # what the last step() updated (graphs.py replays exactly that)
        self._last_tables = []
        self._host_step = 0

    # ------------------------------------------------------------------------------------------
    @property
    def _dense_done(self):
        return max(self._dense_count, default=0)

    def zero_grad(self, set_to_none: bool = True):
        for owner in self._tables:
            owner._stash = None
        for p in self._dense:
            if p.grad is not None:
                if set_to_none:
                    p.grad = None
                else:
                    p.grad.zero_()

    def _sync_hyper(self):
        """Pick up edits of ``param_groups[0]`` (LR schedulers write ``lr`` there)."""
        grp = self.param_groups[0]
        for k in self._FIXED:
            cur = tuple(grp[k]) if isinstance(getattr(self, k), tuple) else float(grp[k])
            if cur != getattr(self, k):
                raise _lib.RlctrError(f"changing {k} after construction is not supported (build a new optimizer)")
        lr = float(grp["lr"])
        if lr != self.lr:
            self.lr = lr
            for owner in self._tables:
                owner._opt.sched.set_lr(lr, owner._opt.host_step + 1)       # steps already taken keep the lr they ran with
            if self._dense_sched is not None:
                self._dense_sched.set_lr(lr, 1)                             # dense parameters never look back

    @torch.no_grad()
    def step(self):
        lib = _lib.load()
        st = _lib.stream()
        self._sync_hyper()
        self._host_step += 1
        self._last_tables = []
        for owner in self._tables:
            opt = owner._opt
            stash = owner._stash
            owner._stash = None
            if stash is None:
                continue                      # torch skips a parameter whose .grad is None: no step, no L2 decay, no counter
            opt.sched.ensure(opt.host_step + 2)
            if hasattr(owner, "_group_update"):  # co-located record (colocated.ColocatedCTR): one update for every member
                owner._group_update(stash, opt, st)
            else:
                t = table_struct(owner.table.data, owner._geom)
                g = _lib.RowGrad(_lib.ptr(stash.staged), _lib.ptr(stash.dlogit), _lib.ptr(stash.sums),
                                 _lib.ptr(stash.extra), stash.fields, stash.flags)
                if stash.peer is not None:           # sharded table: the owner reads every rank's gradient buffers
                    g.world, g.n_per_rank = stash.peer["world"], stash.peer["n_per_rank"]
                    for name in ("staged", "dlogit", "sums", "extra"):
                        ptrs = stash.peer[name]
                        if ptrs is not None:
                            arr = getattr(g, "peer_" + name)
                            for r, ptr_ in enumerate(ptrs):
                                arr[r] = ptr_
                ws_bytes = lib.rlctr_rows_ws_bytes(stash.n)
                ws = owner._rows_ws(ws_bytes)
                opt.rows_update(stash.sorted_ids, stash.sorted_slots, stash.n, g, t, ws, ws_bytes, st, type(owner).__name__,
                                dict(owner._meta(stash.n // stash.fields, stash.fields), extra=stash.extra is not None,
                                     staged=stash.staged is not None, stamp=opt.lazy,
                                     from_stage=getattr(stash, "stage", None) is not None),
                                stage=getattr(stash, "stage", None))
            _lib.check(lib.rlctr_step_advance(_lib.ptr(opt.step), 1, st), "rlctr_step_advance")
            opt.host_step += 1
            self._last_tables.append(owner)
            if opt.lazy:
                opt.dirty = True
                if self.mode == "dense":
                    opt.flush(owner.table.data)
        # ---- replicated dense parameters
        live = [p for p in self._dense if p.grad is not None]
        self._last_live = live
        if live:
            dev = live[0].device
            if self._dense_steps is None:
                self._dense_steps = torch.zeros(max(len(self._dense), 1), dtype=torch.int32, device=dev)
                self._dense_sched = self._dense_schedule(dev)
            self._dense_sched.ensure(self._dense_done + 2)
            grads = []
            for p in live:
                if self._dense_state.get(p) is None:
                    self._dense_state[p] = self._dense_new(p)
                grads.append(p.grad.contiguous())
            for lo in range(0, len(live), _lib.RLCTR_DENSE_MAX):          # one launch per group of tensors (foreach)
                grp, gg = live[lo:lo + _lib.RLCTR_DENSE_MAX], grads[lo:lo + _lib.RLCTR_DENSE_MAX]
                k = len(grp)
                idx = (C.c_int32 * k)(*[self._dense_index[p] for p in grp])
                self._dense_launch(lib, grp, gg, idx, st)
                _lib.check(lib.rlctr_steps_advance(_lib.ptr(self._dense_steps), idx, k, st), "rlctr_steps_advance")
            self._note_dense(live)

    def _note_dense(self, live):
        for p in live:
            self._dense_count[self._dense_index[p]] += 1

    def flush(self):
        for owner in self._tables:
            owner.flush()


def _ptrs(xs):
    return (C.c_void_p * len(xs))(*[x.data_ptr() for x in xs])


class Adam(_RowOptimizer):
    """Differences from ``torch.optim.Adam`` that remain: one parameter group; ``amsgrad`` / ``maximize`` / ``capturable``
    are not offered.  What is kept (each one tested): a parameter without a gradient is skipped and its step counter does not
    advance (tables: no stashed backward -> no step, no L2 decay for that iteration); every dense parameter has its own step
    counter (torch's ``state[p]['step']``), so one that receives its first gradient late starts at step 1; ``param_groups[0]
    ['lr']`` may be edited between steps."""

    _FIXED = ("betas", "eps", "weight_decay")

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, mode="lazy"):
        params = list(params)
        self.lr, self.betas, self.eps, self.weight_decay = float(lr), tuple(betas), float(eps), float(weight_decay)
        self._setup(params, mode, dict(lr=self.lr, betas=self.betas, eps=self.eps, weight_decay=self.weight_decay))

    def _table_state(self, data, geom):
        return TableAdamState(data, geom, self.lr, self.betas, self.eps, self.weight_decay, self.mode)

    def _dense_schedule(self, dev):
        return AdamSchedule(self.lr, self.betas, dev)

    def _dense_new(self, p):
        return (torch.zeros_like(p.data), torch.zeros_like(p.data))

    def _dense_launch(self, lib, grp, grads, idx, st):
        _lib.check(lib.rlctr_dense_adam_multi(_ptrs([p.data for p in grp]), _ptrs(grads),
                                              _ptrs([self._dense_state[p][0] for p in grp]),
                                              _ptrs([self._dense_state[p][1] for p in grp]),
                                              (C.c_int64 * len(grp))(*[p.numel() for p in grp]), len(grp),
                                              _lib.ptr(self._dense_sched.tensor), _lib.ptr(self._dense_steps), idx,
                                              self.betas[0], self.betas[1], self.eps, self.weight_decay, st),
                   "rlctr_dense_adam_multi")


class Adagrad(_RowOptimizer):
    """``torch.optim.Adagrad(params, lr, lr_decay, weight_decay, initial_accumulator_value, eps)`` with torch's numbers
    (``_single_tensor_adagrad``): at a parameter's own step t, ``clr = lr / (1 + (t - 1) * lr_decay)``, ``g += weight_decay
    * p``, ``s += g * g``, ``p -= clr * g / (sqrt(s) + eps)``; ``s`` starts at ``initial_accumulator_value``.  Under the
    reference's dense semantics every table row takes a step every step (rows no sample touched: ``g = weight_decay * p``).

    ``mode``: 'lazy' (default) gives those numbers with O(touched rows) traffic -- with ``weight_decay == 0`` an untouched row
    is exactly unchanged by a dense step, so no catch-up or flush is ever launched; with ``weight_decay > 0`` the missed
    steps are replayed when a row is touched and by ``flush()``.  'dense' replays every row every step (the literal
    reference work).  The table's state sum lives in the record's exp_avg block; table rows use the SFU sqrt / reciprocal
    (DESIGN.md), dense parameters IEEE sqrt and division.

    Differences from ``torch.optim.Adagrad``: one parameter group; ``maximize``, ``foreach``, ``fused``, ``differentiable``
    and sparse gradients are not offered; ``eps == 0`` with ``initial_accumulator_value == 0`` raises ``ValueError`` (torch
    writes 0/0 = NaN into every row no sample touched).  What is kept: ``param_groups[0]['lr']`` may be edited between steps
    (steps already taken keep the lr they ran with); the other hyper-parameters are fixed after construction; a parameter
    without a gradient is skipped and its step counter does not advance; every dense parameter has its own step counter."""

    _FIXED = ("lr_decay", "weight_decay", "initial_accumulator_value", "eps")

    def __init__(self, params, lr=1e-2, lr_decay=0, weight_decay=0, initial_accumulator_value=0, eps=1e-10, mode="lazy"):
        if not 0.0 <= lr:
            raise ValueError(f"Invalid learning rate: {lr}")
        if not 0.0 <= lr_decay:
            raise ValueError(f"Invalid lr_decay value: {lr_decay}")
        if not 0.0 <= weight_decay:
            raise ValueError(f"Invalid weight_decay value: {weight_decay}")
        if not 0.0 <= initial_accumulator_value:
            raise ValueError(f"Invalid initial_accumulator_value value: {initial_accumulator_value}")
        if not 0.0 <= eps:
            raise ValueError(f"Invalid epsilon value: {eps}")
        if eps == 0 and initial_accumulator_value == 0:
            raise ValueError("eps == 0 with initial_accumulator_value == 0 divides 0 by 0 on every row no sample touched "
                             "(torch.optim.Adagrad writes NaN there): give one of them a positive value")
        if mode not in ("lazy", "dense"):
            raise ValueError(f"Invalid mode: {mode!r} ('lazy' or 'dense')")
        params = list(params)
        self.lr, self.lr_decay, self.weight_decay = float(lr), float(lr_decay), float(weight_decay)
        self.initial_accumulator_value, self.eps = float(initial_accumulator_value), float(eps)
        self._setup(params, mode, dict(lr=self.lr, lr_decay=self.lr_decay, weight_decay=self.weight_decay,
                                       initial_accumulator_value=self.initial_accumulator_value, eps=self.eps))

    def _table_state(self, data, geom):
        return TableAdagradState(data, geom, self.lr, self.lr_decay, self.weight_decay, self.initial_accumulator_value,
                                 self.eps, self.mode)

    def _dense_schedule(self, dev):
        return AdagradSchedule(self.lr, self.lr_decay, dev)

    def _dense_new(self, p):
        return torch.full_like(p.data, self.initial_accumulator_value)

    def _dense_launch(self, lib, grp, grads, idx, st):
        _lib.check(lib.rlctr_dense_adagrad_multi(_ptrs([p.data for p in grp]), _ptrs(grads),
                                                 _ptrs([self._dense_state[p] for p in grp]),
                                                 (C.c_int64 * len(grp))(*[p.numel() for p in grp]), len(grp),
                                                 _lib.ptr(self._dense_sched.tensor), _lib.ptr(self._dense_steps), idx,
                                                 self.eps, self.weight_decay, st),
                   "rlctr_dense_adagrad_multi")
