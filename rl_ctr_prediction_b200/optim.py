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


class _RowOptimizer(torch.optim.Optimizer):
    """The step loop shared by :class:`Adam` and :class:`Adagrad`: embedding tables (parameters created by :mod:`.p_model`,
    :mod:`.colocated`, :mod:`.sharded`) get a table state (:mod:`.tables`) that owns the catch-up, row-update and flush
    launches; every other parameter is a replicated dense tensor updated by one multi-tensor launch per step.  A subclass
    provides ``_FIXED`` (hyper-parameters fixed after construction), ``_TORCH_KEYS`` (torch's other group keys, at the values
    implemented), ``_STATE_KEYS`` (torch's names of a parameter's state), ``_table_state``, ``_dense_schedule``, ``_dense_new``,
    ``_dense_blocks`` and ``_dense_launch``.

    It is a ``torch.optim.Optimizer`` with ONE parameter group, so torch's LR schedulers drive it: they edit
    ``param_groups[0]['lr']``, which the next step (or graph replay, :mod:`.graphs`) picks up.  ``state_dict()`` /
    ``load_state_dict()`` save and restore the whole optimizer state exactly (see :meth:`state_dict`)."""

    _FIXED = ()
    _TORCH_KEYS = {}
    _STATE_KEYS = ()
    _EVERY_PARAM = False              # True: every parameter has a state entry from construction on (torch.optim.Adagrad)

    def _setup(self, params, mode, defaults):
        if not params:
            raise ValueError("optimizer got an empty parameter list")
        self.mode = mode
        super().__init__(params, dict(defaults, **self._TORCH_KEYS))
        params = self.param_groups[0]["params"]
        self._tables, self._dense = [], []
        self._slots = []                                # per parameter index: (table owner, None) or (None, dense index)
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
                self._slots.append((owner, None))
                self._tables.append(owner)
            else:
                self._slots.append((None, len(self._dense)))
                self._dense.append(p)
        self._dense_state = {}
        self._dense_index = {p: i for i, p in enumerate(self._dense)}
        self._dense_count = [0] * len(self._dense)      # host mirror of the per-parameter device step counters
        self._dense_steps = None                        # int32 [len(dense)] on the device
        self._dense_sched = None
        self._last_live = []                            # what the last step() updated (graphs.py replays exactly that)
        self._last_tables = []
        self._host_step = 0

    def add_param_group(self, param_group):
        if self.param_groups:
            raise _lib.RlctrError(f"{type(self).__name__} supports one parameter group: pass every parameter in one list, "
                                  "or build one optimizer per group")
        super().add_param_group(param_group)

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
        for k, v in self._TORCH_KEYS.items():
            if grp.get(k) != v:
                raise _lib.RlctrError(f"changing {k} after construction is not supported ({k}={v!r} is what is implemented)")
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

    def _captured(self):
        """The addresses a captured step reads (step scalars, schedule tables, dense state): a graph holding other ones is
        stale and is captured again (graphs.py).  ``load_state_dict`` writes in place, but a schedule that has to grow for a
        later step is reallocated."""
        out = []
        for owner in self._tables:
            out += [owner._opt.step.data_ptr(), owner._opt.sched.tensor.data_ptr()]
        if self._dense_sched is not None:
            out += [self._dense_steps.data_ptr(), self._dense_sched.tensor.data_ptr()]
        for p in self._dense:
            st = self._dense_state.get(p)
            out += [t.data_ptr() for t in self._dense_blocks(st)] if st is not None else [0]
        return tuple(out)

    # ---- checkpoints ------------------------------------------------------------------------------------------------
    @staticmethod
    def _geometry(owner):
        g = owner._geom
        return {"n_rows": int(owner.feature_nums), "used": g.used, "row_stride": g.row_stride, "kind": owner._record_kind}

    def state_dict(self):
        """torch's structure: ``{"state": {i: {...}}, "param_groups": [{...hyper-parameters, "params": [0..n-1]}]}``, ``i`` the
        parameter's position in ``param_groups[0]["params"]`` (the order passed to the constructor).

        A dense parameter's entry is torch's own (``step``: float32 0-d CPU tensor, and ``exp_avg`` / ``exp_avg_sq`` or
        ``sum``): an optimizer over dense parameters only exchanges checkpoints with ``torch.optim.Adam`` /
        ``torch.optim.Adagrad`` both ways.  An embedding table's entry is specific to this library: ``step`` (int), its state
        over the used columns as float32 ``[feature_nums, used]`` tensors in the table's column order (row-sharded tables:
        gathered, the same on every rank and at every world size; every rank must call this), and ``geometry``, which
        ``load_state_dict`` checks.  Lazy tables are flushed first (as ``model.state_dict()`` does): the later steps of the run
        take the same bits whether or not this is called."""
        grp = self.param_groups[0]
        packed = {k: v for k, v in grp.items() if k != "params"}
        packed["params"] = list(range(len(grp["params"])))
        state = {}
        for i, (owner, j) in enumerate(self._slots):
            if owner is not None:
                step = owner._opt.host_step
                if step == 0 and not self._EVERY_PARAM:
                    continue
                ent = {"step": step}
                ent.update(owner._opt_export())
                ent["geometry"] = self._geometry(owner)
            else:
                step = self._dense_count[j]
                if step == 0 and not self._EVERY_PARAM:
                    continue
                p = self._dense[j]
                st = self._dense_state.get(p)
                st = self._dense_new(p) if st is None else st
                ent = {"step": torch.tensor(float(step), dtype=torch.float32)}
                ent.update((k, t.detach().clone()) for k, t in zip(self._STATE_KEYS, self._dense_blocks(st)))
            state[i] = ent
        return {"state": state, "param_groups": [packed]}

    def _check_state(self, state_dict):
        """Every refusal of ``load_state_dict``, before anything is written.  Returns (saved group, entry or None per index)."""
        cls = type(self).__name__
        groups = state_dict["param_groups"]
        if len(groups) != len(self.param_groups):
            raise ValueError("loaded state dict has a different number of parameter groups")
        saved = groups[0]
        for k in self._FIXED:
            if k not in saved:
                raise _lib.RlctrError(f"param_groups[0] has no {k!r}: the checkpoint is not {cls}'s state")
        if len(saved["params"]) != len(self.param_groups[0]["params"]):
            raise ValueError("loaded state dict contains a parameter group that doesn't match the size of optimizer's group")
        entries = [state_dict["state"].get(pid) for pid in saved["params"]]
        for i, (ent, (owner, j)) in enumerate(zip(entries, self._slots)):
            if ent is None:
                continue
            want = {"step", *self._STATE_KEYS} | ({"geometry"} if owner is not None else set())
            if set(ent) != want:
                if owner is not None and "geometry" not in ent:
                    raise _lib.RlctrError(f"state[{i}] is a dense parameter's state, but parameter {i} is an embedding table")
                if owner is None and "geometry" in ent:
                    raise _lib.RlctrError(f"state[{i}] is an embedding table's state, but parameter {i} is a dense tensor")
                raise _lib.RlctrError(f"state[{i}] has the keys {sorted(ent)}: not {cls}'s state ({sorted(want)})")
            step = float(ent["step"])
            if not (step >= 0 and step == int(step)):
                raise _lib.RlctrError(f"state[{i}]['step'] is {step}: a step count is a whole number >= 0")
            if owner is not None:
                geo = self._geometry(owner)
                if ent["geometry"] != geo:
                    raise _lib.RlctrError(f"state[{i}]['geometry'] is {ent['geometry']}, but this table's is {geo}: a table "
                                          "state loads into a table of the same kind and geometry only")
                shape = (geo["n_rows"], geo["used"])
            else:
                shape = tuple(self._dense[j].shape)
            for k in self._STATE_KEYS:
                if tuple(ent[k].shape) != shape:
                    raise _lib.RlctrError(f"state[{i}][{k!r}] has the shape {tuple(ent[k].shape)}, parameter {i} needs {shape}")
        for k in self._FIXED:
            cur = getattr(self, k)
            val = tuple(float(v) for v in saved[k]) if isinstance(cur, tuple) else float(saved[k])
            if val != cur:
                raise _lib.RlctrError(f"param_groups[0][{k!r}] is {saved[k]!r} in the checkpoint and {cur!r} here: construct "
                                      f"the optimizer with {k}={saved[k]!r} to resume from it")
        for k, v in self._TORCH_KEYS.items():
            if k in saved and saved[k] != v:
                raise _lib.RlctrError(f"param_groups[0][{k!r}] is {saved[k]!r} in the checkpoint: only {k}={v!r} is "
                                      "implemented")
        float(saved["lr"])
        return saved, entries

    def load_state_dict(self, state_dict):
        """Resume from :meth:`state_dict` (or, for dense parameters, from torch's own optimizer of the same class): every
        refusal comes before the first write, so a refused load leaves the optimizer and every table as they were.  Fixed
        hyper-parameters must equal the constructed ones; ``lr`` and any other group key (a scheduler's ``initial_lr``) are
        taken from the checkpoint.  ``mode`` is not part of the state: any mode loads any state of its class.  Everything is
        written in place (a captured graph keeps its addresses), every table row ends settled at the saved step, and a
        parameter without an entry starts afresh.  The model's own ``load_state_dict`` may come before or after this."""
        saved, entries = self._check_state(state_dict)
        grp = self.param_groups[0]
        grp.update((k, v) for k, v in saved.items() if k != "params")
        self.lr = float(grp["lr"])
        steps = []
        for ent, (owner, j) in zip(entries, self._slots):
            step = int(float(ent["step"])) if ent is not None else 0
            steps.append(step)
            if owner is None:
                continue
            owner.flush()                       # what the previous state still owes the rows belongs to them
            owner._opt_load({k: ent[k] for k in self._STATE_KEYS} if ent is not None else None, step)
            owner._opt.sched.set_lr(self.lr, step + 1, force=True)  # rows past the saved step may hold lrs edited after it
        dense = [(ent, j, step) for ent, (owner, j), step in zip(entries, self._slots, steps) if owner is None]
        if any(ent is not None for ent, _, _ in dense) and self._dense_steps is None:
            dev = self._dense[0].device
            self._dense_steps = torch.zeros(len(self._dense), dtype=torch.int32, device=dev)
            self._dense_sched = self._dense_schedule(dev)
        for ent, j, step in dense:
            p = self._dense[j]
            st = self._dense_state.get(p)
            if ent is not None and st is None:
                st = self._dense_state[p] = self._dense_new(p)
            if st is not None:
                fresh = self._dense_blocks(self._dense_new(p))
                for k, t, t0 in zip(self._STATE_KEYS, self._dense_blocks(st), fresh):
                    t.copy_(ent[k] if ent is not None else t0)
            self._dense_count[j] = step
        if self._dense_steps is not None:
            self._dense_steps.copy_(torch.tensor(self._dense_count, dtype=torch.int32))
            self._dense_sched.set_lr(self.lr, 1, force=True)
            self._dense_sched.ensure(self._dense_done + 2)
        self._host_step = max(steps, default=0)


def _ptrs(xs):
    return (C.c_void_p * len(xs))(*[x.data_ptr() for x in xs])


class Adam(_RowOptimizer):
    """A ``torch.optim.Optimizer``.  Differences from ``torch.optim.Adam`` that remain: one parameter group (a second one
    raises); ``amsgrad`` / ``maximize`` / ``capturable`` / ``foreach`` / ``fused`` / ``differentiable`` /
    ``decoupled_weight_decay`` keep their default values (editing one raises); a step replayed by :mod:`.graphs`
    (``GraphedTrainStep``, ``GraphedCallable``) does not call ``step()``, so step hooks and an LR scheduler's count of
    optimizer steps see the eager steps only (the scheduler's ``lr`` edits still reach the replays); an embedding table's
    ``state_dict()`` entry is this library's own (see :meth:`_RowOptimizer.state_dict`).  What is kept (each one tested): a
    parameter without a gradient is skipped and its step counter does not advance (tables: no stashed backward -> no step, no
    L2 decay for that iteration); every dense parameter has its own step counter (torch's ``state[p]['step']``), so one that
    receives its first gradient late starts at step 1; ``param_groups[0]['lr']`` may be edited between steps, so torch's LR
    schedulers work (one that edits ``betas``, as ``OneCycleLR`` / ``CyclicLR`` with ``cycle_momentum=True`` do, raises at
    the next step); ``state_dict()`` / ``load_state_dict()`` resume a run bit for bit, and a dense parameter's entry is
    torch's own."""

    _FIXED = ("betas", "eps", "weight_decay")
    _TORCH_KEYS = dict(amsgrad=False, maximize=False, foreach=None, capturable=False, differentiable=False, fused=None,
                       decoupled_weight_decay=False)
    _STATE_KEYS = ("exp_avg", "exp_avg_sq")

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

    def _dense_blocks(self, st):
        return st

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

    A ``torch.optim.Optimizer``.  Differences from ``torch.optim.Adagrad``: one parameter group (a second one raises);
    ``maximize``, ``foreach``, ``fused``, ``differentiable`` keep their default values (editing one raises) and sparse gradients
    are not offered; ``eps == 0`` with ``initial_accumulator_value == 0`` raises ``ValueError`` (torch writes 0/0 = NaN into
    every row no sample touched); graph replays do not call ``step()`` (step hooks and a scheduler's step count see the eager
    steps only); an embedding table's ``state_dict()`` entry is this library's own.  What is kept: ``param_groups[0]['lr']``
    may be edited between steps (steps already taken keep the lr they ran with), so torch's LR schedulers work; the other
    hyper-parameters are fixed after construction; a parameter without a gradient is skipped and its step counter does not
    advance; every dense parameter has its own step counter; as in torch, every parameter has a state entry from construction
    on, and a dense parameter's entry is torch's own."""

    _FIXED = ("lr_decay", "weight_decay", "initial_accumulator_value", "eps")
    _TORCH_KEYS = dict(maximize=False, foreach=None, differentiable=False, fused=None)
    _STATE_KEYS = ("sum",)
    _EVERY_PARAM = True

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

    def _dense_blocks(self, st):
        return (st,)

    def _dense_launch(self, lib, grp, grads, idx, st):
        _lib.check(lib.rlctr_dense_adagrad_multi(_ptrs([p.data for p in grp]), _ptrs(grads),
                                                 _ptrs([self._dense_state[p] for p in grp]),
                                                 (C.c_int64 * len(grp))(*[p.numel() for p in grp]), len(grp),
                                                 _lib.ptr(self._dense_sched.tensor), _lib.ptr(self._dense_steps), idx,
                                                 self.eps, self.weight_decay, st),
                   "rlctr_dense_adagrad_multi")
