"""Fused-row embedding tables: the HBM layout behind the drop-in model classes.

The reference keeps a first-order ``nn.Embedding(N, 1)`` and a latent ``nn.Embedding(N, D)`` (FFM:
F of them) and gathers each separately (src/models/p_model.py:14,34,38,69,76-78,263,267).  Here
one id owns ONE 16-byte aligned row (include/rlctr.h "fused row"):

    LR      [w]                                   row_stride 1
    FM      [w, v_0 .. v_{D-1}, pad]              row_stride = 16 floats (one 64 B DRAM block) for D <= 15
    FFM     [T_0 | T_1 | .. | T_{F-1} | w | pad]  row_stride = round4(F*D + 1)

so a field costs one aligned 128-bit-chunked read instead of two (or F+1) sector-straddling ones.
``state_dict()`` / ``load_state_dict()`` convert to and from the reference's keys and shapes.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import torch

from . import _lib


def round4(n: int) -> int:
    return (n + 3) // 4 * 4


def row_floats(used: int) -> int:
    """Floats per fused row.  Rows that fit in 64 bytes are padded to exactly 64 B and are therefore
    64-byte aligned: ncu shows HBM serves a random access in 64 B blocks (two 32 B sectors), so a 48 B row at
    a 48 B pitch straddles two blocks two times out of three and costs ~107 B of DRAM traffic per access
    (profiles/r1_ncu_top_kernels.md); a 64 B row costs exactly 64.  Wider rows span several blocks anyway
    and only keep the 16 B alignment the 128-bit loads need."""
    n = round4(used)
    return 16 if n <= 16 else n


@dataclass(frozen=True)
class Geometry:
    n_rows: int
    row_stride: int
    lin_col: int
    emb_col: int
    dim: int
    pitch: int = 0            # floats between rows; 0 = row_stride.  3*row_stride: [p | exp_avg | exp_avg_sq] records
    block: int = 0            # floats between the p / exp_avg / exp_avg_sq blocks of a record; 0 = row_stride.  A co-located
                              # record (colocated.py) keeps each block in its own 128-byte line: row_stride 24, block 32, pitch 96
    stamp_at: int = -1        # >= 0: the lazy-Adam stamp's column, chosen by whoever laid the record out (colocated.py)
    offset: int = 0           # floats from the start of the record to this view's column 0: a member's stand-alone view of a wide
                              # co-located record (colocated.py), whose own row starts at its first chunk

    @property
    def row_pitch(self):
        return self.pitch or self.row_stride

    @property
    def block_floats(self):
        return self.block or self.row_stride

    @property
    def has_state(self):
        return self.row_pitch >= 3 * self.block_floats

    @property
    def used(self):
        return max(self.lin_col + 1, self.emb_col + self.dim, 1)

    @property
    def stamp_col(self):
        """Float offset inside the row record where the lazy-Adam stamp lives (-1: separate array).  LR records are
        [w | m | v | stamp]; a row of at most 16 floats whose last active 16-byte chunk has a padding column keeps the
        stamp there; anything else (full rows, wide FFM rows) uses a separate int32 array."""
        if not self.has_state:
            return -1
        if self.stamp_at >= 0:
            return self.stamp_at
        if self.row_stride == 1:
            return 3 if self.row_pitch >= 4 else -1
        if self.row_stride <= 16 and self.used % 4 != 0:
            return self.used
        return -1

    def with_state(self):
        """The trainable layout: Adam's exp_avg / exp_avg_sq interleaved with the row (one contiguous record)."""
        pitch = 4 if self.row_stride == 1 else 3 * self.row_stride
        return Geometry(self.n_rows, self.row_stride, self.lin_col, self.emb_col, self.dim, pitch)

    def rows_only(self, n_rows=None):
        return Geometry(self.n_rows if n_rows is None else n_rows, self.row_stride, self.lin_col, self.emb_col, self.dim, 0)

    @staticmethod
    def lr(n):
        return Geometry(n, 1, 0, 0, 0)

    @staticmethod
    def fm(n, d, with_linear=True):
        if with_linear:
            return Geometry(n, row_floats(1 + d), 0, 1, d)
        return Geometry(n, row_floats(d), -1, 0, d)

    @staticmethod
    def ffm(n, f, d):
        return Geometry(n, round4(f * d + 1), f * d, 0, f * d)


def table_struct(data: torch.Tensor, g: Geometry) -> _lib.Table:
    p = _lib.ptr(data)
    return _lib.Table(p + 4 * g.offset if g.offset else p, g.n_rows, g.row_stride, g.lin_col, g.emb_col, g.dim, g.row_pitch)


class AdamSchedule:
    """The two Python-double scalars torch.optim.Adam derives per step (torch/optim/adam.py
    ``_single_tensor_adam``): step_size = lr / (1 - beta1^t) and sqrt(1 - beta2^t), tabulated
    for t = 0..len-1 and kept on the device so the step index can be a device scalar.

    ``set_lr(lr, from_step)`` re-tabulates the entries t >= from_step IN PLACE (same device address: a captured CUDA graph
    keeps working): an ``lr`` edited through ``param_groups`` -- an LR scheduler, or the reference's ``learning_rate += 1e-4``
    per epoch -- takes effect from that step on, while the lazy replay of earlier steps still sees the lr they ran with."""

    def __init__(self, lr, betas, device, length=8192):
        self.lr, self.betas, self.device = float(lr), (float(betas[0]), float(betas[1])), device
        self.length = 0
        self.tensor = None
        self.rows = [(0.0, 1.0)]
        self.ensure(length)

    def _row(self, t):
        b1, b2 = self.betas
        return (self.lr / (1 - b1 ** t), (1 - b2 ** t) ** 0.5)

    def _upload(self, lo, hi):
        part = torch.tensor(self.rows[lo:hi], dtype=torch.float64).to(torch.float32).to(self.device)
        self.tensor[lo:hi].copy_(part)

    def ensure(self, steps: int):
        if steps < self.length:
            return False
        n = max(steps + 1, 2 * self.length, 1024)
        self.rows.extend(self._row(t) for t in range(len(self.rows), n))
        self.tensor = torch.tensor(self.rows, dtype=torch.float64).to(torch.float32).to(self.device).contiguous()
        self.length = n
        return True

    def set_lr(self, lr, from_step: int):
        if float(lr) == self.lr:
            return
        self.lr = float(lr)
        lo = max(int(from_step), 1)
        for t in range(lo, self.length):
            self.rows[t] = self._row(t)
        if lo < self.length:
            self._upload(lo, self.length)


def _key(entry, tag):
    return entry if tag is None else f"{entry}[{tag}]"


class _TableState:
    """What the training step asks of a table's optimizer state, whatever the optimizer: bring the batch's rows up to date
    (``catchup``), apply the step to the rows the batch touched (``rows_update`` / ``group_update``) and settle every row
    (``flush``).  A subclass names its C entry points and provides ``struct()``, ``lazy`` and ``lookup_on``."""

    _CATCHUP = _ROWS = _GROUP = _FLUSH = None
    catchup_ids_ok = False            # rlctr_rows_catchup_ids (batch-order catch-up of co-located records) serves this state

    def catchup(self, t, sorted_ids, n, tag, meta):
        """Replay the L2-only steps the rows of the sorted view missed (lazy state with rows behind ``step``)."""
        if not (self.lazy and self.dirty):
            return
        lib = _lib.load()
        _lib.call(self._CATCHUP, getattr(lib, self._CATCHUP), _lib.ptr(sorted_ids), n, C.byref(t), C.byref(self.struct()),
                  _lib.stream(), key=_key(self._CATCHUP, tag), meta=meta)

    def rows_update(self, sorted_ids, sorted_slots, n, grad, t, ws, ws_bytes, st, tag, meta, stage=None):
        lib = _lib.load()
        _lib.call(self._ROWS, getattr(lib, self._ROWS), _lib.ptr(sorted_ids), _lib.ptr(sorted_slots), n, C.byref(grad),
                  C.byref(t), C.byref(self.struct(stage)), _lib.ptr(ws), ws_bytes, st, key=_key(self._ROWS, tag), meta=meta)

    def group_update(self, sorted_ids, sorted_slots, n, t, members, n_members, sums, sums_pitch, fields, world, slot_of, ws,
                     ws_bytes, st, tag, meta):
        lib = _lib.load()
        _lib.call(self._GROUP, getattr(lib, self._GROUP), _lib.ptr(sorted_ids), _lib.ptr(sorted_slots), n, C.byref(t),
                  C.byref(self.struct()), members, n_members, _lib.ptr(sums), sums_pitch, fields, world, _lib.ptr(slot_of),
                  _lib.ptr(ws), ws_bytes, st, key=_key(self._GROUP, tag), meta=meta)

    def flush(self, data: torch.Tensor):
        """Replay the L2-only steps every row missed."""
        if not self.lazy or not self.dirty:
            return
        lib = _lib.load()
        t = table_struct(data, self.geom)
        _lib.call(self._FLUSH, getattr(lib, self._FLUSH), C.byref(t), C.byref(self.struct()), 0, self.geom.n_rows, _lib.stream(),
                  meta={"rs": self.geom.row_stride, "n_rows": self.geom.n_rows})
        self.dirty = False


class TableAdamState(_TableState):
    """exp_avg / exp_avg_sq / per-row stamp for one fused table, plus the lazy-exact bookkeeping.

    mode 'lazy'   (default): rows are brought up to date when touched (rlctr_rows_catchup) and by
                  ``flush()`` before anything reads the whole table -- same numbers as the reference's
                  dense Adam (SURVEY N3) with O(touched rows) HBM traffic per step.
    mode 'dense'  : every step also streams the whole table (the literal reference work).
    mode 'sparse' : untouched rows are left alone (numerically NOT the reference; SURVEY H1 mode C).
    """

    _CATCHUP, _ROWS, _GROUP, _FLUSH = "rlctr_rows_catchup", "rlctr_rows_adam", "rlctr_group_rows_adam", "rlctr_adam_flush"
    catchup_ids_ok = True

    def __init__(self, param: torch.Tensor, geom: Geometry, lr, betas, eps, weight_decay, mode):
        assert mode in ("lazy", "dense", "sparse")
        self.geom, self.mode = geom, mode
        dev = param.device
        rs = geom.row_stride
        if geom.has_state:            # [p | exp_avg | exp_avg_sq] records: the state lives inside the table's rows
            blk = geom.block_floats
            param[:, blk:3 * blk].zero_()
            self.exp_avg = param[:, blk:blk + rs]
            self.exp_avg_sq = param[:, 2 * blk:2 * blk + rs]
        else:
            self.exp_avg = torch.zeros_like(param)
            self.exp_avg_sq = torch.zeros_like(param)
        self.stamp_col = -1
        if mode == "sparse":
            self.stamp = None
        elif geom.stamp_col >= 0:
            self.stamp = None                         # the stamp rides inside the record (tables.Geometry.stamp_col)
            self.stamp_col = geom.stamp_col
            param[:, self.stamp_col].zero_()
        else:
            self.stamp = torch.zeros(geom.n_rows, dtype=torch.int32, device=dev)
        self.step = torch.zeros(1, dtype=torch.int32, device=dev)     # completed steps (device scalar)
        self.host_step = 0
        self.sched = AdamSchedule(lr, betas, dev)
        self.betas, self.eps, self.weight_decay = betas, float(eps), float(weight_decay)
        self.dirty = False           # True while some rows lag behind `step` (lazy mode)

    @property
    def lazy(self):
        """True when untouched rows are owed their L2-only steps (modes 'lazy' and 'dense')."""
        return self.stamp is not None or self.stamp_col >= 0

    def struct(self, stage=None) -> _lib.Adam:
        return _lib.Adam(self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(), _lib.ptr(self.stamp),
                         _lib.ptr(self.sched.tensor), _lib.ptr(self.step), self.sched.length, self.stamp_col,
                         self.betas[0], self.betas[1], self.eps, self.weight_decay, _lib.ptr(stage))

    @property
    def lookup_ok(self):
        """rlctr_rows_lookup serves this table: LR records, or vector rows of at most 16 floats whose stamp rides inside the
        record (or that carry no stamp at all: mode 'sparse')."""
        g = self.geom
        return g.has_state and (g.row_stride == 1 or (g.row_stride <= 16 and self.stamp is None))

    @property
    def lookup_on(self):
        """Whether the training step takes the lookup path (rlctr_rows_lookup -> streamed forward -> update from the stage)
        instead of catch-up -> gather by id -> update.  Measured on one B200 (profiles/r2_rows_lookup_ab.md): the lookup
        path moves fewer DRAM bytes (812 vs 950 MB per FM step) but the replay it has to do is instruction-bound, not
        memory-bound, and the extra staging writes make the step ~6 % SLOWER (1.75 vs 1.65 ms) -- so it is off unless
        RLCTR_LOOKUP=1.  Kept because it is the owner-pushes-rows form of the sharded lookup."""
        return self.lookup_ok and os.environ.get("RLCTR_LOOKUP", "0") == "1"



class AdagradSchedule:
    """torch.optim.Adagrad's per-step scalar ``clr = lr / (1 + (t - 1) * lr_decay)`` (torch/optim/adagrad.py
    ``_single_tensor_adagrad``), a Python double cast to fp32, tabulated for t = 0..len-1 on ``device`` (entry 0 unused).
    ``ensure`` / ``set_lr`` behave as :class:`AdamSchedule`'s: an lr edit re-tabulates t >= from_step in place."""

    def __init__(self, lr, lr_decay, device, length=8192):
        self.lr, self.lr_decay, self.device = float(lr), float(lr_decay), device
        self.length = 0
        self.tensor = None
        self.rows = [0.0]
        self.ensure(length)

    def _row(self, t):
        return self.lr / (1 + (t - 1) * self.lr_decay)

    def ensure(self, steps: int):
        if steps < self.length:
            return False
        n = max(steps + 1, 2 * self.length, 1024)
        self.rows.extend(self._row(t) for t in range(len(self.rows), n))
        self.tensor = torch.tensor(self.rows, dtype=torch.float64).to(torch.float32).to(self.device).contiguous()
        self.length = n
        return True

    def set_lr(self, lr, from_step: int):
        if float(lr) == self.lr:
            return
        self.lr = float(lr)
        lo = max(int(from_step), 1)
        for t in range(lo, self.length):
            self.rows[t] = self._row(t)
        if lo < self.length:
            self.tensor[lo:self.length].copy_(torch.tensor(self.rows[lo:self.length], dtype=torch.float64).to(torch.float32))


class TableAdagradState(_TableState):
    """torch.optim.Adagrad's state_sum for one fused table: it lives in the record's exp_avg block; the exp_avg_sq block is
    never read or written.

    With ``weight_decay == 0`` a dense Adagrad step leaves every row no sample touched exactly as it was, so mode 'lazy' keeps
    no stamps and never launches a catch-up or a flush: it is the reference's numbers with O(touched rows) traffic as it stands.
    With ``weight_decay > 0`` (and in mode 'dense') the rows carry stamps like :class:`TableAdamState`'s and the missed L2-only
    steps g = wd * p are replayed (rlctr_adagrad_catchup / rlctr_adagrad_flush); mode 'dense' flushes after every step."""

    _CATCHUP, _ROWS, _GROUP, _FLUSH = "rlctr_adagrad_catchup", "rlctr_rows_adagrad", "rlctr_group_rows_adagrad", "rlctr_adagrad_flush"
    lookup_on = False                 # the lookup path (RLCTR_LOOKUP) is Adam's

    def __init__(self, param: torch.Tensor, geom: Geometry, lr, lr_decay, weight_decay, initial_accumulator_value, eps, mode):
        assert mode in ("lazy", "dense")
        self.geom, self.mode = geom, mode
        dev = param.device
        rs = geom.row_stride
        if geom.has_state:
            blk = geom.block_floats
            self.state_sum = param[:, blk:blk + rs]
        else:
            self.state_sum = torch.empty_like(param)
        self.state_sum.fill_(float(initial_accumulator_value))
        self.stamp, self.stamp_col = None, -1
        if geom.stamp_col >= 0:
            param[:, geom.stamp_col].zero_()          # a previous optimizer's stamp: a padding column of p again
        if weight_decay != 0 or mode == "dense":
            if geom.stamp_col >= 0:
                self.stamp_col = geom.stamp_col
            else:
                self.stamp = torch.zeros(geom.n_rows, dtype=torch.int32, device=dev)
        self.step = torch.zeros(1, dtype=torch.int32, device=dev)
        self.host_step = 0
        self.sched = AdagradSchedule(lr, lr_decay, dev)
        self.eps, self.weight_decay = float(eps), float(weight_decay)
        self.dirty = False

    @property
    def lazy(self):
        """True when untouched rows are owed their L2-only steps (weight_decay > 0, or mode 'dense')."""
        return self.stamp is not None or self.stamp_col >= 0

    def struct(self, stage=None) -> _lib.Adagrad:
        assert stage is None
        return _lib.Adagrad(self.state_sum.data_ptr(), _lib.ptr(self.stamp), _lib.ptr(self.sched.tensor), _lib.ptr(self.step),
                            self.sched.length, self.stamp_col, self.eps, self.weight_decay)
