"""Co-located records: several CTR models trained on the same id stream share ONE row record per id.

The reference trains its models one after the other on the same encoded batches (``get_model`` names in
src/main/pretrain_main.py:25-45, loop :96-103) and the RL ensemble scores M of them on every sample
(src/all_main/main.py:183-271); each keeps its own ``nn.Embedding`` tables, so a batch costs one random gather and one
random optimizer update PER MODEL per (sample, field).  On the B200 a random HBM access costs the same whether it returns
4 or 128 bytes (profiles/r2_rowprobe.md: ~30-36 G accesses/s for 16 .. 128-byte rows), so the models' parameters of one id
are laid side by side in one record

    [ FM: w v0..v9 | LR: w ][ DeepFM: w v0..v9 | stamp ] (pad)     p block       (one 128-byte line)
    [ exp_avg of the same columns                       ] (pad)     exp_avg block
    [ exp_avg_sq                                        ] (pad)     exp_avg_sq block

and one gather (rlctr_group_fwd), one catch-up (rlctr_rows_catchup) and one update (rlctr_group_rows_adam) serve all of
them: 13 random line operations per (sample, field) and step instead of 23 for LR + FM + DeepFM.  Members may be any of the
FM-row models of ``get_model`` (FFM's rows are wider than a line): LR, FM, DeepFM, WideAndDeep, FNN, InnerPNN, OuterPNN, DCN
and AFM -- at D = 10 two vector members and LR fill one line (e.g. LR + FM + FNN, DeepFM + InnerPNN, FM + AFM).  A member with
a dense tail computes its logit with its own ``_tail(z_table, rows)`` from the group's gather, so its tower, cross network or
attention (and the dropout masks they draw from the member's own counter) are those of the stand-alone model.  Each member
keeps the chunk alignment of its stand-alone row, so its logits and its updated parameters are bit-identical to the
stand-alone model's (tests/test_gpu_colocated.py, tests/test_gpu_colocated_tails.py).

    lr, fm, dfm = (get_model(name, ...).to(dev) for name in ("LR", "FM", "DeepFM"))
    group = colocate([lr, fm, dfm])                       # re-homes the three tables into one; the members stay usable
    opt = optim.Adam(group.parameters(), lr=1e-3, weight_decay=1e-5)
    losses = group.train_step(x, y, opt)                  # float32 [3]: one BCE loss per member
    fm(x); fm.state_dict()                                # inference and reference-keyed checkpoints work per member
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import torch
import torch.nn as nn

from . import _lib
from . import p_model as Model
from .tables import Geometry, round4, table_struct


# the member kinds of one joint record: an FM-type row [w?, v_0 .. v_{D-1}] (or LR's scalar) and a logit the group step computes
MEMBER_KINDS = (Model.LR, Model.FM, Model.DeepFM, Model.WideAndDeep, Model.FNN, Model.InnerPNN, Model.OuterPNN, Model.DCN,
                Model.AFM)


# 1: the group's catch-up works from the ids in batch order and the sort of the batch runs on a side stream (see train_step);
# 0 (default): sort first, catch-up over the sorted run heads.  The two leave the same bits in the table.  Measured A/B on one
# B200 (C2 step): 1.347 ms sorted, 1.422 ms with the sort off the critical path -- the batch-order catch-up with its claim
# atomics and the concurrent sort cost more than the 66 us of sorting they hide, so it stays an option.
UNSORTED_CATCHUP = os.environ.get("RLCTR_GROUP_UNSORTED_CATCHUP", "0") != "0"


@dataclass(slots=True)
class GroupStash:
    """What a group step leaves for the optimizer: the sorted view, the joint column sums and each member's gradient side.  The
    last four fields describe the row-sharded group's exchange (sharded.ShardedGroup); their defaults are the one-device group's."""
    sorted_ids: torch.Tensor
    sorted_slots: torch.Tensor
    n: int
    fields: int
    sums: torch.Tensor
    dlogit: list                       # per member: dL/dlogit [B], or None when it rides in the sums row
    extra: list                        # per member: the tower-input gradient rows, or None
    sums_pitch: int = 0                # floats between two samples' sums rows; 0 = the record's row_stride
    world: int = 1
    slot_of: torch.Tensor | None = None    # routed exchange: the global slot at every receive position
    extra_pitch: list | None = None        # per member: floats between two rows of ``extra``; None = 0 for every member


def labels(y):
    """(int64 labels, None) or (None, float32 labels): what rlctr_bce_fwd_bwd reads."""
    y = y.reshape(-1).contiguous()
    return (y, None) if y.dtype == torch.int64 else (None, y.float())


def loss_head(m, logit, rows, y, loss, ws, dl=None, scale=1.0):
    """Sigmoid + BCE of one model's logit and their gradient (rlctr_bce_fwd_bwd).  ``logit`` [B] is the table part (None for a
    model without one); with tower rows [B, F*D] the logit is ``m._tail(logit, rows)``, run under autograd on a detached leaf.
    ``scale`` multiplies dL/dlogit and the bias gradient before the tail's backward (1/G in a row-sharded step: the gradient of
    the GLOBAL mean loss).  ``y``: :func:`labels`; the loss goes to the device address ``loss``, dL/dlogit to ``dl`` (allocated
    when None), the bias gradient to ``m.bias.grad``.  Returns (dL/dlogit [B], the gradient of ``rows`` or None)."""
    lib = _lib.load()
    src = rows if rows is not None else logit
    B, dev = src.shape[0], src.device
    dl = torch.empty(B, dtype=torch.float32, device=dev) if dl is None else dl
    bias = getattr(m, "bias", None)
    dbias = torch.empty(1, dtype=torch.float32, device=dev) if bias is not None else None
    z = leaf = None
    if rows is None:
        zz = logit
    else:
        leaf = rows.detach().requires_grad_(True)
        z = m._tail(logit.view(B, 1) if logit is not None else None, leaf)
        zz = z.detach().reshape(-1).contiguous()
    # (the head's own sum of dlogit is the bias gradient: the same block partition and tree as the stand-alone backward's
    # rlctr_sigmoid_bwd sum -- the same bits, one launch less)
    _lib.check(lib.rlctr_bce_fwd_bwd(_lib.ptr(zz), _lib.ptr(y[0]), _lib.ptr(y[1]), None, loss, _lib.ptr(dl), _lib.ptr(dbias),
                                     _lib.ptr(ws), B, _lib.stream()), "rlctr_bce_fwd_bwd")
    if scale != 1.0:
        dl.mul_(scale)
        if dbias is not None:
            dbias.mul_(scale)
    grad = None
    if z is not None:
        z.backward(dl.view_as(z))
        grad = leaf.grad.contiguous()
    if bias is not None:
        bias.grad = dbias
    return dl, grad


MAX_LINES = 4                          # a joint row spans at most four 128-byte lines (rlctr.h RLCTR_GROUP_MAX_FLOATS)


def _layout(members, max_lines=1):
    """Columns of the joint row.  Vector members (FM-type rows: [w, v_0 .. v_{D-1}]) take consecutive 16-byte aligned blocks
    with their stand-alone layout; scalar members (LR) fill the padding columns those blocks leave, else open a new chunk.  The
    row, with the stamp in the last active chunk, must fit ``max_lines`` 128-byte lines (1..4); a one-line record holds only
    members whose stand-alone rows are at most 16 floats.  Returns ([(lin_col, emb_col, dim)] per member, used columns)."""
    if not 1 <= max_lines <= MAX_LINES:
        raise ValueError(f"max_lines must be 1..{MAX_LINES} (128-byte lines per joint row), got {max_lines}")
    cols, taken, nxt = [None] * len(members), set(), 0
    for i, m in enumerate(members):
        g = m._geom
        if g.row_stride == 1:
            continue
        if g.lin_col > g.emb_col or g.row_stride > 36:
            raise _lib.RlctrError(f"{type(m).__name__}: FFM rows (F field-aware blocks) cannot be co-located")
        if g.row_stride > 16 and max_lines == 1:
            raise _lib.RlctrError(f"{type(m).__name__}: rows of {g.row_stride} floats do not fit the one-line record (32 floats) "
                                  "beside the stamp of members with rows of at most 16 floats; pass max_lines=2..4 for a wider record")
        lin = nxt + g.lin_col if g.lin_col >= 0 else -1
        cols[i] = (lin, nxt + g.emb_col, g.dim)
        for c in ([lin] if lin >= 0 else []) + list(range(nxt + g.emb_col, nxt + g.emb_col + g.dim)):
            taken.add(c)
        nxt += round4(g.used)
    for i, m in enumerate(members):
        if m._geom.row_stride != 1:
            continue
        free = [c for c in range(nxt) if c not in taken]
        c = free[0] if free else nxt
        if not free:
            nxt += 4
        taken.add(c)
        cols[i] = (c, 0, 0)
    used = max(taken) + 1
    if used % 4 == 0:
        used += 1                       # the stamp needs a padding column in the last active chunk: open one
    rs = round4(used + 1)
    if rs > 32 * max_lines:
        need = (rs + 31) // 32
        hint = f"; pass max_lines={need}" if need <= MAX_LINES else f" (at most {MAX_LINES} lines, {32 * MAX_LINES} floats)"
        raise _lib.RlctrError(f"co-located record of {rs} floats wider than {32 * max_lines} floats "
                              f"({'one 128-byte line' if max_lines == 1 else f'{max_lines} 128-byte lines'}): too many members{hint}")
    return cols, used


def _wide(members, used):
    """The record needs the wide kernels: more than one line, or a member whose stand-alone row is wider than 16 floats."""
    return round4(used + 1) > 32 or any(m._geom.row_stride > 16 for m in members)


def _record(n_rows, used):
    """Geometry of the joint record over ``used`` columns (stamp at ``used``).  One line: [p | exp_avg | exp_avg_sq] each in its own
    128-byte line (block 32, pitch 96).  Wider: the three blocks packed (block = row_stride), the pitch rounded up to whole lines,
    so every record and its p block start on a line: fewer lines per record than line-aligned blocks (DESIGN §6b)."""
    rs = round4(used + 1)
    if rs <= 32:
        return Geometry(n_rows, rs, -1, 0, used, pitch=96, block=32, stamp_at=used)
    return Geometry(n_rows, rs, -1, 0, used, pitch=(3 * rs + 31) // 32 * 32, block=rs, stamp_at=used)


def _member_view(m, rec, col, wide):
    """Member ``m``'s view of the joint record ``rec`` at columns ``col`` = (lin, emb, dim).  One-line records keep the joint row
    (the one-line gather serves it); a wide record gives each member its stand-alone row -- from its first chunk, its own
    row_stride, the joint pitch -- so that its own forward, state_dict and load_state_dict work on rows of at most 36 floats."""
    lin, emb, dim = col
    if not wide:
        return Geometry(rec.n_rows, rec.row_stride, lin, emb, dim, pitch=rec.row_pitch, block=rec.block_floats)
    if dim == 0:                                             # LR: its one column
        return Geometry(rec.n_rows, 1, 0, 0, 0, pitch=rec.row_pitch, block=rec.block_floats, offset=lin)
    base = (emb if lin < 0 else min(lin, emb)) // 4 * 4
    return Geometry(rec.n_rows, m._geom.row_stride, lin - base if lin >= 0 else -1, emb - base, dim, pitch=rec.row_pitch,
                    block=rec.block_floats, offset=base)


class _GroupStep:
    """The parts of a group step that do not depend on where the joint table lives, shared by ColocatedCTR (one device) and
    sharded.ShardedGroup (row-sharded).  The class provides ``members``, ``_cols``, ``_geom``, ``table``, ``_meta``,
    ``_reduce_ws``, ``_rows_ws``, ``_global_struct()`` (the table as the gathers read it) and ``_UPDATE_TAG``."""

    def _member_structs(self, B, F, dev, train, pctr=None):
        """The members' views for rlctr_group_fwd.  logits[i]: the table part of member i's logit (bias + first order + FM
        term), None for a member that has none (FNN, InnerPNN, OuterPNN, DCN: no linear column, no bias); rows[i]: the tower
        input [B, pitch] of a member with a dense tail, else None."""
        arr = (_lib.Member * len(self.members))()
        logits, rows = [], []
        for i, (m, (lin, emb, dim)) in enumerate(zip(self.members, self._cols)):
            s = arr[i]
            s.lin_col, s.emb_col, s.dim = lin, emb, dim
            s.flags = _lib.RLCTR_FM_TERM if m._fm_term else 0
            bias = getattr(m, "bias", None)
            s.bias = _lib.ptr(bias.data) if bias is not None else None
            tail = hasattr(m, "_tail")
            table_part = lin >= 0 or bias is not None or m._fm_term
            z = torch.empty(B, dtype=torch.float32, device=dev) if table_part and (train or tail) else None
            logits.append(z)
            s.logit = _lib.ptr(z)
            if pctr is not None and not tail:
                s.pctr, s.pctr_stride = pctr.data_ptr() + 4 * i, pctr.shape[1]
            r = None
            if tail:
                pitch = round4(F * dim)                      # 16-byte aligned pitch: the tower's first GEMM fetches it by TMA
                r = torch.empty(B, pitch, dtype=torch.float32, device=dev)
                s.rows_out, s.rows_pitch = r.data_ptr(), pitch
            rows.append(r)
        return arr, logits, rows

    def _pctr(self, x, key):
        """pCTR of every member on one gather: float32 [B, M] (column m = ``members[m](x)``)."""
        lib = _lib.load()
        B, F = x.shape
        out = torch.empty(B, len(self.members), dtype=torch.float32, device=x.device)
        arr, logits, rows = self._member_structs(B, F, x.device, False, pctr=out)
        t = self._global_struct()
        _lib.call("rlctr_group_fwd", lib.rlctr_group_fwd, _lib.ptr(x), C.byref(t), arr, len(self.members), None, 0, B, F,
                  _lib.stream(), key=key, meta=self._meta(B, F))
        for i, m in enumerate(self.members):
            if rows[i] is not None:
                z = logits[i].view(B, 1) if logits[i] is not None else None
                out[:, i:i + 1] = torch.sigmoid(m._tail(z, rows[i][:, :F * self._cols[i][2]]))
        return out

    def _heads(self, F, logits, rows, y, scale=1.0):
        """Every member's loss head (:func:`loss_head`) on the group's gather, the dense gradients set afresh.  Returns the losses
        float32 [M], and dL/dlogit and the tower-input gradient (or None) per member."""
        for p in self.parameters():
            p.grad = None
        losses = torch.empty(len(self.members), dtype=torch.float32, device=self.table.device)
        ws = self._reduce_ws(self.table.device)
        dlogits, extras = [], []
        for i, m in enumerate(self.members):
            r = rows[i][:, :F * self._cols[i][2]] if rows[i] is not None else None
            dl, grad = loss_head(m, logits[i], r, y, losses.data_ptr() + 4 * i, ws, scale=scale)
            dlogits.append(dl)
            extras.append(grad)
        return losses, dlogits, extras

    def _group_update(self, stash, opt_state, st):
        """The optimizer step for the joint table: rlctr_group_rows_adam / rlctr_group_rows_adagrad."""
        lib = _lib.load()
        M = len(self.members)
        arr = (_lib.Member * M)()
        pitches = stash.extra_pitch or [0] * M
        for i, (m, (lin, emb, dim)) in enumerate(zip(self.members, self._cols)):
            s = arr[i]
            s.lin_col, s.emb_col, s.dim = lin, emb, dim
            s.flags = _lib.RLCTR_FM_TERM if m._fm_term else 0
            s.dlogit = _lib.ptr(stash.dlogit[i])
            s.extra = _lib.ptr(stash.extra[i])
            s.extra_pitch = pitches[i]
        ws_bytes = lib.rlctr_rows_ws_bytes(stash.n)
        ws = self._rows_ws(ws_bytes)
        opt_state.group_update(stash.sorted_ids, stash.sorted_slots, stash.n, table_struct(self.table.data, self._geom), arr, M,
                               stash.sums, stash.sums_pitch, stash.fields, stash.world, stash.slot_of, ws, ws_bytes, st,
                               self._UPDATE_TAG, self._meta(stash.n // stash.fields, stash.fields))


class ColocatedCTR(_GroupStep, Model._TableModel):
    """``colocate(models)``: LR / FM-type drop-in models (``MEMBER_KINDS``) over one joint table.  The group owns the table,
    its lazy-exact Adam state and the training step; the members keep ``forward`` (inference), ``state_dict`` /
    ``load_state_dict`` (reference keys) and their dense parameters."""

    _kind = "group"
    _UPDATE_TAG = None

    def __init__(self, models, max_lines=1):
        super().__init__()
        models = list(models)
        if not 1 <= len(models) <= _lib.RLCTR_GROUP_MAX:
            raise ValueError(f"a co-located group holds 1..{_lib.RLCTR_GROUP_MAX} models")
        for m in models:
            # LR / FM: table only; the others: logit = m._tail(table part or None, gathered rows)
            if type(m) not in MEMBER_KINDS or m.__dict__.get("_group") is not None:
                raise _lib.RlctrError(f"{type(m).__name__} cannot join a co-located group "
                                      f"({', '.join(k.__name__ for k in MEMBER_KINDS)}; once)")
        n_rows = {m._geom.n_rows for m in models}
        devs = {m.table.device for m in models}
        if len(n_rows) != 1 or len(devs) != 1:
            raise ValueError("members of a group share the vocabulary (feature_nums) and the device")
        dev = devs.pop()
        if dev.type != "cuda":
            raise _lib.RlctrError("move the models to the CUDA device before co-locating them")
        self.feature_nums = n_rows.pop()
        cols, used = _layout(models, max_lines)
        self._geom = _record(self.feature_nums, used)
        wide = _wide(models, used)
        joint = torch.zeros(self.feature_nums, self._geom.row_pitch, dtype=torch.float32, device=dev)
        with torch.no_grad():
            for m, (lin, emb, dim) in zip(models, cols):
                m.flush()                                    # settle what a previous optimizer still owes the stand-alone table
                g, src = m._geom, m.table.data
                if lin >= 0:
                    joint[:, lin].copy_(src[:, g.lin_col])
                if dim:
                    joint[:, emb:emb + dim].copy_(src[:, g.emb_col:g.emb_col + dim])
        self.table = nn.Parameter(joint)
        self.table._rlctr_owner = self
        self._opt, self._stash, self._ws = None, None, {}
        self._sort_stream, self._claim = None, None
        self._cols, self._max_lines = cols, max_lines
        for m, col in zip(models, cols):
            m.table = self.table                             # shared Parameter: the member's view of the joint record
            m._geom = _member_view(m, self._geom, col, wide)
            m._opt, m._stash = None, None
            m.__dict__["_group"] = self                      # not a sub-module of the member: no cycle in parameters()
        self.members = nn.ModuleList(models)

    # ---- nn.Module plumbing ---------------------------------------------------------------------------------------
    def _apply(self, fn, recurse=True):
        out = super()._apply(fn, recurse)
        self.table._rlctr_owner = self
        return out

    def _ref_items(self):
        return []

    def _save_to_state_dict(self, destination, prefix, keep_vars):
        self.flush()                                         # the members write the reference keys from the joint table

    def _load_from_state_dict(self, state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys, error_msgs):
        self.flush()

    def _meta(self, B, F):
        g = self._geom
        return {"model": "+".join(type(m).__name__ for m in self.members), "B": B, "F": F, "rs": g.row_stride, "dim": g.dim,
                "n_rows": g.n_rows, "lin": False, "members": [(type(m).__name__, c[2]) for m, c in zip(self.members, self._cols)]}

    def _global_struct(self):
        """The joint table as the gathers read it (one device: the table itself)."""
        return table_struct(self.table.data, self._geom)

    @torch.no_grad()
    def forward(self, x):
        """pCTR of every member on one gather: float32 [B, M] (column m = ``members[m](x)``)."""
        x = Model._check_ids(x)
        self.flush()
        return self._pctr(x, "rlctr_group_fwd[infer]")

    # ---- the training step ---------------------------------------------------------------------------------------
    def train_step(self, x, y, optimizer):
        """One step of src/main/pretrain_main.py:96-102 for EVERY member on the batch (x, y): sort -> catch-up -> one gather ->
        per member: (tower,) sigmoid + BCE and their gradient -> one segment-reduce + Adam over the joint record -> dense Adam.
        Returns the members' losses, float32 [M] on the device."""
        lib = _lib.load()
        opt = self._opt
        if opt is None:
            raise _lib.RlctrError("build rl_ctr_prediction_b200.optim.Adam(group.parameters(), ...) (or optim.Adagrad) before "
                                  "training the group")
        x = Model._check_ids(x)
        B, F = x.shape
        dev, st, g = x.device, _lib.stream(), self._geom
        y = labels(y)
        t = table_struct(self.table.data, g)
        # The sorted view is needed by the scatter at the END of the step only: with the catch-up working from the ids in batch
        # order (rlctr_rows_catchup_ids: a claim bit per row tells the occurrences of an id apart) the sort runs on its own
        # stream -- a parallel branch of a captured step -- beside catch-up, gather and tower instead of in front of them.
        side = None
        if UNSORTED_CATCHUP and opt.catchup_ids_ok and opt.lazy and opt.stamp_col >= 0 and 5 <= (g.used + 3) // 4 <= 8:
            cur = torch.cuda.current_stream(dev)
            side = self._sort_stream
            if side is None or side.device != dev:
                side = self._sort_stream = torch.cuda.Stream(device=dev)
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                sid, sslot = Model.sort_ids(x, g.n_rows)
            if opt.dirty:
                a = opt.struct()
                cb = lib.rlctr_rows_claim_bytes(g.n_rows)
                if self._claim is None or self._claim.numel() < cb or self._claim.device != dev:
                    self._claim = torch.empty(cb, dtype=torch.uint8, device=dev)
                _lib.call("rlctr_rows_catchup_ids", lib.rlctr_rows_catchup_ids, _lib.ptr(x), x.numel(), C.byref(t), C.byref(a),
                          _lib.ptr(self._claim), cb, st, key="rlctr_rows_catchup[group]", meta=self._meta(B, F))
        else:
            sid, sslot = Model.sort_ids(x, g.n_rows)
            opt.catchup(t, sid, x.numel(), "group", self._meta(B, F))
        M = len(self.members)
        arr, logits, rows = self._member_structs(B, F, dev, True)
        sums = torch.empty(B, g.row_stride, dtype=torch.float32, device=dev)
        _lib.call("rlctr_group_fwd", lib.rlctr_group_fwd, _lib.ptr(x), C.byref(t), arr, M, _lib.ptr(sums), 0, B, F, st,
                  key="rlctr_group_fwd[train]", meta=self._meta(B, F))
        losses, dlogits, extras = self._heads(F, logits, rows, y)
        self._stash = GroupStash(sorted_ids=sid, sorted_slots=sslot, n=B * F, fields=F, sums=sums, dlogit=dlogits, extra=extras)
        if side is not None:
            torch.cuda.current_stream(dev).wait_stream(side)     # join: the scatter reads the sorted view
        optimizer.step()
        return losses


def colocate(models, max_lines=1) -> ColocatedCTR:
    """One joint record per id for ``models`` (``MEMBER_KINDS``, up to RLCTR_GROUP_MAX, same vocabulary and device).  The record
    takes the fewest 128-byte lines that hold the members' columns, up to ``max_lines`` (1..4).  The default, one line, is the
    measured layout; a group that needs more lines is refused with a message that names the ``max_lines`` it needs."""
    return ColocatedCTR(models, max_lines)
