"""Drop-in CTR model classes over the sm_100a hot path (mirror of the reference's
``src/models/p_model.py``: same class names, constructor signatures, ``forward(x: int64[B,F]) ->
pctr float32[B,1]`` and ``state_dict`` keys / shapes -- SURVEY section 8b).

What differs is everything underneath: parameters live in one fused-row table per model
(:mod:`.tables`), ``forward`` is one fused gather + interaction kernel, and ``backward`` does not
materialise a dense ``[N, D]`` gradient: it leaves ``(sorted ids, dlogit, saved sums)`` on the
module for :class:`rl_ctr_prediction_b200.optim.Adam`, whose ``step()`` runs the
sort / segment-reduce / fused-Adam kernel.  There is no CPU path: calling a model with host
tensors raises.
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.nn as nn

from . import _lib
from .tables import Geometry, table_struct
from . import mlp as _mlp


class RowsStash:
    """What one backward pass leaves for the optimizer (struct rlctr_rowgrad + the sorted ids)."""
    __slots__ = ("sorted_ids", "sorted_slots", "n", "dlogit", "sums", "extra", "staged", "fields", "flags", "peer", "stage")

    def __init__(self, **kw):
        for k in self.__slots__:
            setattr(self, k, kw.get(k))


def _check_ids(x: torch.Tensor) -> torch.Tensor:
    if not x.is_cuda:
        raise _lib.RlctrError("rl_ctr_prediction_b200 models run on a CUDA (sm_100a) device only; "
                              "move the features with .to(device) -- there is no CPU fallback")
    if x.dtype != torch.int64:
        x = x.long()
    if x.dim() != 2:
        raise ValueError("features must be int64 [batch, field_nums]")
    return x.contiguous()


_SORT_CACHE = {"key": None, "x": None, "out": None}


def sort_ids(x: torch.Tensor, n_rows: int):
    """(sorted_ids u32[n], sorted_slots u32[n]) of the flattened ids: rlctr_sort_ids.

    One batch usually feeds several models (LR, FM, DeepFM... train on the same features, and the RL
    step scores M models on them): the sorted view of a batch is computed once and shared while the SAME
    tensor object (unmodified: same ``_version``) is presented again for a table of the same height.  The
    cache keeps that tensor alive, so its storage cannot be recycled under the key."""
    key = (id(x), x._version, x.data_ptr(), tuple(x.shape), int(n_rows))
    if _SORT_CACHE["key"] == key and _SORT_CACHE["x"] is x:
        return _SORT_CACHE["out"]
    out = _sort_ids(x, n_rows)
    _SORT_CACHE.update(key=key, x=x, out=out)
    return out


def _sort_ids(x: torch.Tensor, n_rows: int):
    lib = _lib.load()
    n = x.numel()
    dev = x.device
    sid = torch.empty(n, dtype=torch.int32, device=dev)
    sslot = torch.empty(n, dtype=torch.int32, device=dev)
    ws_bytes = lib.rlctr_sort_ws_bytes(n, n_rows)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    _lib.call("rlctr_sort_ids", lib.rlctr_sort_ids, _lib.ptr(x), n, n_rows, _lib.ptr(sid), _lib.ptr(sslot), _lib.ptr(ws),
              ws_bytes, _lib.stream(), meta={"n": n})
    return sid, sslot


def lookup_rows(module, sorted_pair, n, fields, gathered=None, world=1, n_per_rank=0, peer_ptrs=None, key=None):
    """The owner-side lookup of a training step (rlctr_rows_lookup): every distinct row of the sorted view is read once,
    brought up to date in registers and written (a) to ``stage`` at its sorted position, for the optimizer, and (b) to the
    sample-ordered ``gathered`` buffer of whoever asked for it.  Returns (stage, gathered)."""
    lib = _lib.load()
    g, opt = module._geom, module._opt
    data = module.table.data
    dev = data.device
    t, a = table_struct(data, g), opt.struct()
    stage = torch.empty(n * lib.rlctr_lookup_stage_floats(C.byref(t)), dtype=torch.float32, device=dev)
    lk = _lib.Lookup(stage.data_ptr(), world if world > 1 else 0, n_per_rank)
    if peer_ptrs is None:
        if gathered is None:
            gathered = module._gathered_rows(n)
        lk.gathered[0] = gathered.data_ptr()
    else:
        for r, p_ in enumerate(peer_ptrs):
            lk.gathered[r] = p_
    ws_bytes = lib.rlctr_rows_ws_bytes(n)
    ws = module._rows_ws(ws_bytes)
    _lib.call("rlctr_rows_lookup", lib.rlctr_rows_lookup, _lib.ptr(sorted_pair[0]), _lib.ptr(sorted_pair[1]), n, C.byref(t),
              C.byref(a), C.byref(lk), _lib.ptr(ws), ws_bytes, _lib.stream(),
              key=key or f"rlctr_rows_lookup[{type(module).__name__}]", meta=dict(module._meta(n // max(fields, 1), fields), n=n))
    return stage, gathered


def gathered_struct(gathered, n, g):
    """``gathered`` as the table the forward kernels stream (ids == NULL: row (b, f) is row b * F + f)."""
    return _lib.Table(gathered.data_ptr(), n, g.row_stride, g.lin_col, g.emb_col, g.dim, g.row_stride)


class _GatherInteract(torch.autograd.Function):
    """ids -> fused gather + first/second order -> (out[B,1], rows[B,F*D] | empty).

    ``out`` is the post-sigmoid pCTR when ``apply_sigmoid`` else the logit.  The table gradient is
    never materialised: backward stashes it in row form on the module (returns None for it)."""

    @staticmethod
    def forward(ctx, module, ids, table, bias, want_rows, apply_sigmoid, sorted_pair, lookup=None):
        lib = _lib.load()
        g = module._geom
        B, F = ids.shape
        dev = ids.device
        need_bwd = sorted_pair is not None
        out = torch.empty(B, 1, dtype=torch.float32, device=dev)
        logit = None if apply_sigmoid else out
        pctr = out if apply_sigmoid else None
        sums = None
        # tower input: rows of F*D floats at a 16-byte aligned pitch, so the first GEMM can fetch them by TMA
        rows_pitch = (F * g.dim + 3) // 4 * 4
        rows = torch.empty(B, rows_pitch, dtype=torch.float32, device=dev) if want_rows else None
        partners = None
        t = table_struct(table, g)
        ids_ptr = _lib.ptr(ids)
        if lookup is not None:                              # training step: the rows were pushed into `gathered` in sample order
            t, ids_ptr = gathered_struct(lookup[1], B * F, g), None
        if module._kind == "ffm":
            if need_bwd:
                partners = torch.empty(B * F, g.row_stride, dtype=torch.float32, device=dev)
            _lib.call("rlctr_ffm_fwd", lib.rlctr_ffm_fwd, _lib.ptr(ids), C.byref(t), _lib.ptr(bias), _lib.ptr(logit),
                      _lib.ptr(pctr), 1, _lib.ptr(partners), B, F, module.latent_dims, _lib.stream(),
                      key="rlctr_ffm_fwd" + ("[train]" if need_bwd else "[infer]"), meta=module._meta(B, F))
        else:
            if need_bwd and module._kind == "fm" and module._fm_term:
                sums = torch.empty(B, g.row_stride, dtype=torch.float32, device=dev)
            flags = _lib.RLCTR_FM_TERM if module._fm_term else 0
            _lib.call("rlctr_embed_fwd", lib.rlctr_embed_fwd, ids_ptr, C.byref(t), _lib.ptr(bias), _lib.ptr(logit),
                      _lib.ptr(pctr), 1, _lib.ptr(sums), _lib.ptr(rows), rows_pitch, B, F, flags, _lib.stream(),
                      key=f"rlctr_embed_fwd[{type(module).__name__}]",
                      meta=dict(module._meta(B, F), sums=sums is not None, rows=want_rows, streamed=lookup is not None))
        hook = getattr(module, "_after_gather", None)       # graphs.GraphedTrainStep: fork point of the captured step
        if hook is not None:
            module._after_gather = None
            hook()
        ctx.module, ctx.sorted_pair, ctx.apply_sigmoid = module, sorted_pair, apply_sigmoid
        ctx.sums, ctx.partners, ctx.shape = sums, partners, (B, F)
        ctx.stage = lookup[0] if lookup is not None else None
        ctx.has_bias = bias is not None
        if apply_sigmoid:
            ctx.save_for_backward(out)
        if rows is None:
            rows = torch.empty(0, device=dev)
            ctx.mark_non_differentiable(rows)
        elif rows_pitch != F * g.dim:
            rows = rows[:, :F * g.dim]                  # [B, F*D] view of the padded buffer (pad columns never read)
        return out, rows

    @staticmethod
    def backward(ctx, gout, grows):
        lib = _lib.load()
        module = ctx.module
        if ctx.sorted_pair is None:
            raise _lib.RlctrError("backward through a forward that ran without gradient bookkeeping")
        if module._opt is None and not getattr(module, "rows_grad_only", False):
            # (set ``model.rows_grad_only = True`` to inspect the row-form gradient -- module._stash -- without an optimizer)
            raise _lib.RlctrError("the embedding table's gradient exists only in row form (sorted ids + per-sample terms) and is "
                                  "consumed by rl_ctr_prediction_b200.optim.Adam(model.parameters(), ...) or optim.Adagrad: build "
                                  "that optimizer before calling backward -- a torch.optim optimizer would silently skip the table "
                                  "(its .grad is never materialised)")
        B, F = ctx.shape
        dev = gout.device
        gout = gout.contiguous()
        dbias = torch.empty(1, dtype=torch.float32, device=dev) if ctx.has_bias else None
        ws = module._reduce_ws(dev)
        if ctx.apply_sigmoid:
            (p,) = ctx.saved_tensors
            dlogit = torch.empty(B, dtype=torch.float32, device=dev)
            _lib.check(lib.rlctr_sigmoid_bwd(_lib.ptr(gout), _lib.ptr(p), _lib.ptr(dlogit), _lib.ptr(dbias),
                                             _lib.ptr(ws), B, _lib.stream()), "rlctr_sigmoid_bwd")
        else:
            dlogit = gout.reshape(B)
            if dbias is not None:
                _lib.check(lib.rlctr_sigmoid_bwd(None, None, _lib.ptr(dlogit), _lib.ptr(dbias), _lib.ptr(ws), B,
                                                 _lib.stream()), "rlctr_sigmoid_bwd")
        if module._stash is not None:
            raise _lib.RlctrError("two backward passes without an optimizer step in between are not supported "
                                  "(the reference loop does one: src/main/pretrain_main.py:100-102)")
        extra = grows.contiguous() if (grows is not None and grows.numel() > 0) else None
        sid, sslot = ctx.sorted_pair
        module._stash = RowsStash(sorted_ids=sid, sorted_slots=sslot, n=B * F, dlogit=dlogit, sums=ctx.sums,
                                  extra=extra, staged=ctx.partners, fields=F,
                                  flags=_lib.RLCTR_STAGED_PARTNER if ctx.partners is not None else 0, stage=ctx.stage)
        return None, None, None, dbias, None, None, None, None


class _TableModel(nn.Module):
    """Shared machinery of the drop-in classes: the fused table, reference-keyed state_dict, the
    lazy-exact optimizer hand-shake."""

    _kind = "fm"          # 'lr' | 'fm' | 'ffm'
    _fm_term = False

    def _init_table(self, geom: Geometry, columns, device=None):
        """columns: list of (first_col, tensor[N, w]) in the reference's creation order."""
        geom = geom.with_state()            # trainable: Adam state interleaved with the row (tables.Geometry)
        self._geom = geom
        dev = torch.device(device) if device is not None else None
        data = torch.zeros(geom.n_rows, geom.row_pitch, dtype=torch.float32, device=dev)
        for col, w in columns:
            # nn.Embedding.reset_parameters == normal_(0, 1), drawn in the reference's creation order:
            # with the default (CPU) construction the same torch.manual_seed gives the reference's values
            if dev is not None and dev.type == "cuda":
                data[:, col:col + w].normal_()
            else:
                data[:, col:col + w].copy_(torch.empty(geom.n_rows, w).normal_())
        self.table = nn.Parameter(data)
        self.table._rlctr_owner = self
        self._opt = None
        self._stash = None
        self._ws = {}

    def _apply(self, fn, recurse=True):
        out = super()._apply(fn, recurse)
        # .to(device) may have replaced the Parameter object; a member of a co-located group shares the group's table
        self.table._rlctr_owner = self.__dict__.get("_group") or self
        self._ws = {}
        return out

    def _meta(self, B, F):
        g = self._geom
        return {"model": type(self).__name__, "B": B, "F": F, "rs": g.row_stride, "dim": g.dim, "n_rows": g.n_rows,
                "lin": g.lin_col >= 0}

    def _reduce_ws(self, dev):
        ws = self._ws.get("reduce")
        if ws is None or ws.device != dev:
            ws = torch.zeros(_lib.RLCTR_REDUCE_WS_BYTES, dtype=torch.uint8, device=dev)
            self._ws["reduce"] = ws
        return ws

    def _rows_ws(self, nbytes):
        """Workspace of the row kernels (heavy-hitter list), kept across steps: no allocation on the step's critical path."""
        ws = self._ws.get("rows")
        if ws is None or ws.numel() < nbytes or ws.device != self.table.device:
            ws = torch.empty(nbytes, dtype=torch.uint8, device=self.table.device)
            self._ws["rows"] = ws
        return ws

    def _gathered_rows(self, n):
        """The sample-ordered lookup buffer [n, row_stride] rlctr_rows_lookup fills (kept per batch size: its padding
        columns are zeroed once and never written)."""
        key = ("gathered", n)
        buf = self._ws.get(key)
        if buf is None:
            buf = torch.zeros(n, self._geom.row_stride, dtype=torch.float32, device=self.table.device)
            self._ws[key] = buf
        return buf

    # ---- reference-keyed state_dict -----------------------------------------------------------
    def _ref_items(self):
        """[(reference key, first column, width)]"""
        raise NotImplementedError

    def flush(self):
        """Make the table equal to what the reference's dense Adam would hold right now."""
        grp = self.__dict__.get("_group")
        if grp is not None:
            return grp.flush()                  # member of a co-located group: the group owns the table and its Adam state
        if self._opt is not None:
            self._opt.flush(self.table.data)

    # ---- optimizer checkpoints (optim._RowOptimizer.state_dict / load_state_dict) --------------------------------------
    @property
    def _record_kind(self):
        """What a checkpointed optimizer state of this table is laid out for, beside its geometry."""
        return self._kind

    def _opt_export(self):
        """The optimizer state of the whole table ({name: float32 [feature_nums, used]}), settled first."""
        self.flush()
        return self._opt.export()

    def _opt_load(self, state, step):
        self._opt.load(self.table.data, state, step)

    def _save_to_state_dict(self, destination, prefix, keep_vars):
        self.flush()
        for name, p in self._parameters.items():
            if name != "table" and p is not None:
                destination[prefix + name] = p if keep_vars else p.detach()
        tab = self.table.detach()
        off = self._geom.offset
        for key, col, w in self._ref_items():
            destination[prefix + key] = tab[:, off + col:off + col + w].clone()

    def _load_from_state_dict(self, state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys,
                              error_msgs):
        self.flush()
        handled = set()
        with torch.no_grad():
            for key, col, w in self._ref_items():
                k = prefix + key
                handled.add(k)
                if k not in state_dict:
                    missing_keys.append(k)
                    continue
                src = state_dict[k]
                if tuple(src.shape) != (self._geom.n_rows, w):
                    error_msgs.append(f"size mismatch for {k}: checkpoint {tuple(src.shape)} vs model "
                                      f"{(self._geom.n_rows, w)}")
                    continue
                off = self._geom.offset + col
                self.table.data[:, off:off + w].copy_(src)
            for name, p in self._parameters.items():
                if name == "table" or p is None:
                    continue
                k = prefix + name
                handled.add(k)
                if k not in state_dict:
                    missing_keys.append(k)
                elif tuple(state_dict[k].shape) != tuple(p.shape):
                    error_msgs.append(f"size mismatch for {k}")
                else:
                    p.data.copy_(state_dict[k])
        if strict:
            for k in state_dict:
                if k.startswith(prefix) and k not in handled:
                    head = k[len(prefix):].split(".", 1)[0]
                    if head not in self._modules:
                        unexpected_keys.append(k)

    # ---- forward plumbing ---------------------------------------------------------------------
    def _run(self, x, want_rows, apply_sigmoid):
        x = _check_ids(x)
        if x.shape[1] != getattr(self, "field_nums", x.shape[1]):
            raise ValueError(f"expected {self.field_nums} fields, got {x.shape[1]}")
        track = torch.is_grad_enabled() and self.table.requires_grad
        sorted_pair = None
        lookup = None
        if self.__dict__.get("_group") is not None:
            # member of a co-located group (colocated.py): inference only -- the group's train_step trains all members at once
            if track and self.training:
                raise _lib.RlctrError("this model is a member of a co-located group: train it with group.train_step(x, y, opt); "
                                      "call the member itself under torch.no_grad() / model.eval()")
            track = False
        if track:
            sorted_pair = sort_ids(x, self._geom.n_rows)
            opt = self._opt
            if opt is not None and opt.lookup_on:
                lookup = lookup_rows(self, sorted_pair, x.numel(), x.shape[1])
            elif opt is not None:
                opt.catchup(table_struct(self.table.data, self._geom), sorted_pair[0], x.numel(), type(self).__name__,
                            self._meta(*x.shape))
        else:
            self.flush()
        bias = getattr(self, "bias", None)
        return _GatherInteract.apply(self, x, self.table, bias, want_rows, apply_sigmoid, sorted_pair, lookup)

    def zero_grad(self, set_to_none: bool = True):
        self._stash = None
        return super().zero_grad(set_to_none)


class LR(_TableModel):
    """p_model.py:9-26  sigma(bias + sum_f w[x_f])."""
    _kind = "lr"

    def __init__(self, feature_nums, output_dim=1, device=None):
        super().__init__()
        assert output_dim == 1
        self.feature_nums = feature_nums
        self._init_table(Geometry.lr(feature_nums), [(0, 1)], device)
        self.bias = nn.Parameter(torch.zeros((output_dim,), device=device))

    def _ref_items(self):
        return [("linear.weight", self._geom.lin_col, 1)]

    def forward(self, x):
        return self._run(x, False, True)[0]


class FM(_TableModel):
    """p_model.py:28-57  sigma(bias + sum_f w[x_f] + 0.5 sum_d[(sum_f v)^2 - sum_f v^2])."""
    _kind = "fm"
    _fm_term = True

    def __init__(self, feature_nums, latent_dims, output_dim=1, device=None):
        super().__init__()
        assert output_dim == 1
        self.feature_nums, self.latent_dims = feature_nums, int(latent_dims)
        g = Geometry.fm(feature_nums, self.latent_dims)
        self._init_table(g, [(g.lin_col, 1), (g.emb_col, g.dim)], device)
        self.bias = nn.Parameter(torch.zeros((output_dim,), device=device))

    def _ref_items(self):
        g = self._geom
        return [("linear.weight", g.lin_col, 1), ("feature_embedding.weight", g.emb_col, g.dim)]

    def forward(self, x):
        return self._run(x, False, True)[0]


class FFM(_TableModel):
    """p_model.py:59-100  sigma(bias + sum_f w[x_f] + sum_{i<j} <T_j[x_i], T_i[x_j]>)."""
    _kind = "ffm"

    def __init__(self, feature_nums, field_nums, latent_dims, output_dim=1, device=None):
        super().__init__()
        assert output_dim == 1
        self.feature_nums, self.field_nums, self.latent_dims = feature_nums, int(field_nums), int(latent_dims)
        g = Geometry.ffm(feature_nums, self.field_nums, self.latent_dims)
        cols = [(g.lin_col, 1)] + [(g.emb_col + t * self.latent_dims, self.latent_dims) for t in range(self.field_nums)]
        self._init_table(g, cols, device)
        self.bias = nn.Parameter(torch.zeros((output_dim,), device=device))

    def _ref_items(self):
        g, D = self._geom, self.latent_dims
        return [("linear.weight", g.lin_col, 1)] + \
               [(f"field_feature_embeddings.{t}.weight", g.emb_col + t * D, D) for t in range(self.field_nums)]

    def forward(self, x):
        return self._run(x, False, True)[0]


def colocate(models, max_lines=1):
    """Re-home LR / FM-type models trained on the same id stream into ONE joint table (colocated.ColocatedCTR) of at most
    ``max_lines`` 128-byte lines per row (1..4)."""
    from .colocated import ColocatedCTR
    return ColocatedCTR(models, max_lines)


def _tower(in_dims: int, device=None) -> nn.Sequential:
    """[in -> 300 -> 200 -> 1], ReLU + Dropout(0.2) after each hidden layer (p_model.py:276-293); Linear
    layers sit at Sequential indices 0, 3, 6 as in the reference's state_dict.  The Linear layers are
    :class:`rl_ctr_prediction_b200.mlp.Linear` (tcgen05 3xTF32 GEMM kernels, same parameters)."""
    mods, d = [], in_dims
    for width in (300, 200):
        mods += [_mlp.Linear(d, width, device=device), nn.ReLU(), nn.Dropout(p=0.2)]
        d = width
    mods.append(_mlp.Linear(d, 1, device=device))
    return _mlp.Tower(*mods)


class DeepFM(FM):
    """p_model.py:256-324  FM logit + MLP(concat_f v_f).  One gather feeds both terms (the reference
    gathers the table twice, :303 and :320)."""

    def __init__(self, feature_nums, field_nums, latent_dims, output_dim=1, device=None):
        super().__init__(feature_nums, latent_dims, output_dim, device)
        self.field_nums = int(field_nums)
        self.mlp = _tower(self.field_nums * self.latent_dims, device)

    def _tail(self, z, rows):
        """Logit [B, 1] from the table part z (bias + first order + FM term, [B, 1]) and the gathered rows [B, F*D]: the one
        definition the stand-alone ``logit`` and a co-located group's step (colocated.py) share."""
        return z + self.mlp(rows)

    def logit(self, x):
        """Pre-sigmoid output [B, 1] (graphs.eager_step feeds it to the fused sigmoid + BCE head)."""
        return self._tail(*self._run(x, True, False))

    def forward(self, x):
        return torch.sigmoid(self.logit(x))


class _PairDots(torch.autograd.Function):
    """rows [B, F*D] -> [E | ip] (InnerPNN tower input, p_model.py:189-194): rlctr_pairdots_fwd / _bwd."""

    @staticmethod
    def forward(ctx, rows, fields, dim):
        lib = _lib.load()
        B, fd = rows.shape
        npair = fields * (fields - 1) // 2
        ld_rows = rows.stride(0) if (rows.stride(1) == 1 and B > 1) else fd
        if not (rows.stride(1) == 1 and (B == 1 or rows.stride(0) >= fd)):
            rows, ld_rows = rows.contiguous(), fd
        pitch = (fd + npair + 3) // 4 * 4                      # 16-byte aligned pitch: the tower's first GEMM reads it by TMA
        out = torch.empty(B, pitch, dtype=torch.float32, device=rows.device)
        _lib.call("rlctr_pairdots_fwd", lib.rlctr_pairdots_fwd, rows.data_ptr(), ld_rows, _lib.ptr(out), pitch, B, fields, dim, 0,
                  _lib.stream(), meta={"B": B})
        ctx.save_for_backward(rows)
        ctx.geom = (fields, dim, ld_rows, pitch)
        return out[:, :fd + npair] if pitch != fd + npair else out

    @staticmethod
    def backward(ctx, gout):
        lib = _lib.load()
        (rows,) = ctx.saved_tensors
        fields, dim, ld_rows, pitch = ctx.geom
        B, fd = rows.shape
        gout = gout.contiguous()
        grows = torch.empty(B, fd, dtype=torch.float32, device=rows.device)
        _lib.call("rlctr_pairdots_bwd", lib.rlctr_pairdots_bwd, rows.data_ptr(), ld_rows, _lib.ptr(gout), gout.shape[1],
                  _lib.ptr(grows), fd, B, fields, dim, 0, _lib.stream(), meta={"B": B})
        return grows, None, None


class WideAndDeep(_TableModel):
    """p_model.py:103-144  sigma(bias + sum_f w[x_f] + MLP(concat_f v_f)): the DeepFM layout without the FM term."""
    _kind = "fm"
    _fm_term = False

    def __init__(self, feature_nums, field_nums, latent_dims, output_dim=1, device=None):
        super().__init__()
        assert output_dim == 1
        self.feature_nums, self.field_nums, self.latent_dims = feature_nums, int(field_nums), int(latent_dims)
        g = Geometry.fm(feature_nums, self.latent_dims)
        self._init_table(g, [(g.lin_col, 1), (g.emb_col, g.dim)], device)          # linear, then embedding (:115,118)
        self.bias = nn.Parameter(torch.zeros((output_dim,), device=device))
        self.mlp = _tower(self.field_nums * self.latent_dims, device)

    def _ref_items(self):
        g = self._geom
        return [("linear.weight", g.lin_col, 1), ("embedding.weight", g.emb_col, g.dim)]

    def _tail(self, z, rows):
        return z + self.mlp(rows)

    def logit(self, x):
        return self._tail(*self._run(x, True, False))

    def forward(self, x):
        return torch.sigmoid(self.logit(x))


class FNN(_TableModel):
    """p_model.py:326-373  sigma(MLP(concat_f v_f)); ``load_embedding`` takes an FM checkpoint (:358-363)."""
    _kind = "fm"
    _fm_term = False

    def __init__(self, feature_nums, field_nums, latent_dims, device=None):
        super().__init__()
        self.feature_nums, self.field_nums, self.latent_dims = feature_nums, int(field_nums), int(latent_dims)
        g = Geometry.fm(feature_nums, self.latent_dims, with_linear=False)
        self._init_table(g, [(g.emb_col, g.dim)], device)
        self.mlp = self._make_tower(device)

    def _make_tower(self, device):
        return _tower(self.field_nums * self.latent_dims, device)

    def _ref_items(self):
        g = self._geom
        return [("feature_embedding.weight", g.emb_col, g.dim)]

    def load_embedding(self, pretrain_params):
        self.flush()
        g = self._geom
        c = g.offset + g.emb_col                 # a member of a wide co-located record: its view starts at g.offset
        with torch.no_grad():
            self.table.data[:, c:c + g.dim].copy_(pretrain_params["feature_embedding.weight"])

    def _tower_input(self, rows):
        return rows

    def _tail(self, z, rows):
        """No first-order term and no bias: the logit is the tower's output alone and z is not read (None in a group)."""
        return self.mlp(self._tower_input(rows))

    def logit(self, x):
        return self._tail(*self._run(x, True, False))

    def forward(self, x):
        return torch.sigmoid(self.logit(x))


class InnerPNN(FNN):
    """p_model.py:146-200  sigma(MLP([concat_f v_f | <v_i, v_j> for i < j]))."""

    def _make_tower(self, device):
        F = self.field_nums
        return _tower(F * self.latent_dims + F * (F - 1) // 2, device)

    def _tower_input(self, rows):
        return _PairDots.apply(rows, self.field_nums, self.latent_dims)


class _FieldSq(torch.autograd.Function):
    """rows [B, F*D] -> [E | D * (sum_f v_f)^2] (OuterPNN tower input, p_model.py:245-251): rlctr_fieldsq_fwd / _bwd."""

    @staticmethod
    def forward(ctx, rows, fields, dim):
        lib = _lib.load()
        rows, ld_rows = _mlp._rows_view(rows)
        B, fd = rows.shape
        pitch = (fd + dim + 3) // 4 * 4
        out = torch.empty(B, pitch, dtype=torch.float32, device=rows.device)
        _lib.call("rlctr_fieldsq_fwd", lib.rlctr_fieldsq_fwd, rows.data_ptr(), ld_rows, _lib.ptr(out), pitch, B, fields, dim,
                  _lib.stream(), meta={"B": B})
        ctx.save_for_backward(rows)
        ctx.geom = (fields, dim, ld_rows)
        return out[:, :fd + dim] if pitch != fd + dim else out
    @staticmethod
    def backward(ctx, gout):
        lib = _lib.load()
        (rows,) = ctx.saved_tensors
        fields, dim, ld_rows = ctx.geom
        B, fd = rows.shape
        gout = gout.contiguous()
        grows = torch.empty(B, fd, dtype=torch.float32, device=rows.device)
        _lib.call("rlctr_fieldsq_bwd", lib.rlctr_fieldsq_bwd, rows.data_ptr(), ld_rows, _lib.ptr(gout), gout.shape[1],
                  _lib.ptr(grows), fd, B, fields, dim, _lib.stream(), meta={"B": B})
        return grows, None, None


class OuterPNN(FNN):
    """p_model.py:202-254  sigma(MLP([concat_f v_f | sum_i (S * K[i]) * S])), S = sum_f v_f.  The reference's ``kernel``
    is a constant ``torch.ones((D, D)).cuda()`` (:236; not a parameter, not in the state_dict -- SURVEY N8), so the product
    term is D * S^2 per dimension; it is kept as a plain attribute for code that inspects it."""

    def __init__(self, feature_nums, field_nums, latent_dims, output_dim=1, device=None):
        super().__init__(feature_nums, field_nums, latent_dims, device)
        self.kernel = torch.ones((self.latent_dims, self.latent_dims), device=device)

    def _make_tower(self, device):
        return _tower(self.latent_dims + self.field_nums * self.latent_dims, device)

    def _tower_input(self, rows):
        return _FieldSq.apply(rows, self.field_nums, self.latent_dims)


class _CrossNet(torch.autograd.Function):
    """x0 [B, F*D], W [L, F*D], Bv [L, F*D] -> x_L (DCN cross network, p_model.py:423-428): rlctr_cross_fwd / _bwd."""

    @staticmethod
    def forward(ctx, rows, W, Bv):
        lib = _lib.load()
        rows, ldx = _mlp._rows_view(rows)
        B, fd = rows.shape
        L = W.shape[0]
        W, Bv = W.detach().contiguous(), Bv.detach().contiguous()
        out = torch.empty(B, fd, dtype=torch.float32, device=rows.device)
        s = torch.empty(B, L, dtype=torch.float32, device=rows.device)
        _lib.call("rlctr_cross_fwd", lib.rlctr_cross_fwd, rows.data_ptr(), ldx, _lib.ptr(W), _lib.ptr(Bv), L, _lib.ptr(out), fd,
                  _lib.ptr(s), B, fd, _lib.stream(), meta={"B": B, "L": L, "fd": fd})
        ctx.save_for_backward(rows, W, Bv, s)
        ctx.ldx = ldx
        return out

    @staticmethod
    def backward(ctx, gout):
        lib = _lib.load()
        rows, W, Bv, s = ctx.saved_tensors
        B, fd = rows.shape
        L = W.shape[0]
        gout = gout.contiguous()
        dev = rows.device
        gx0 = torch.empty(B, fd, dtype=torch.float32, device=dev)
        dw, db = torch.empty_like(W), torch.empty_like(Bv)
        ws_bytes = lib.rlctr_cross_ws_bytes(B, fd, L)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        _lib.call("rlctr_cross_bwd", lib.rlctr_cross_bwd, rows.data_ptr(), ctx.ldx, _lib.ptr(W), _lib.ptr(Bv), _lib.ptr(s), L,
                  _lib.ptr(gout), gout.shape[1], _lib.ptr(gx0), fd, _lib.ptr(dw), _lib.ptr(db), B, fd, _lib.ptr(ws), ws_bytes,
                  _lib.stream(), meta={"B": B, "L": L, "fd": fd})
        return gx0, dw, db


class DCN(_TableModel):
    """p_model.py:376-435  sigma(Linear([cross_L(x0) | DN(x0)])), x0 = concat_f v_f: 5 cross layers
    ``x_{l+1} = x0 <x_l, w_l> + b_l + x_l`` (one kernel, forward and backward) beside the [300, 200] deep net (tcgen05 tower).
    state_dict keys are the reference's: ``feature_embedding.weight, DN.{0,3}.*, cross_net_w.{l}.weight (1, F*D),
    cross_net_b.{l} (F*D,), linear.*``."""
    _kind = "fm"
    _fm_term = False

    def __init__(self, feature_nums, field_nums, latent_dims, output_dim=1, device=None):
        super().__init__()
        assert output_dim == 1
        self.feature_nums, self.field_nums, self.latent_dims = feature_nums, int(field_nums), int(latent_dims)
        g = Geometry.fm(feature_nums, self.latent_dims, with_linear=False)
        self._init_table(g, [(g.emb_col, g.dim)], device)                               # :387
        fd = self.field_nums * self.latent_dims
        self.num_neural_layers = 5                                                      # :394
        mods, d = [], fd
        for width in (300, 200):                                                        # :396-400 (ends in ReLU, Dropout)
            mods += [_mlp.Linear(d, width, device=device), nn.ReLU(), nn.Dropout(p=0.2)]
            d = width
        self.DN = _mlp.Tower(*mods)
        self.cross_net_w = nn.ModuleList([nn.Linear(fd, output_dim, bias=False, device=device)
                                          for _ in range(self.num_neural_layers)])     # :409-411
        self.cross_net_b = nn.ParameterList([nn.Parameter(torch.zeros((fd,), device=device))
                                             for _ in range(self.num_neural_layers)])  # :415-417
        self.linear = _mlp.Linear(200 + fd, output_dim, device=device)                  # :419

    def _ref_items(self):
        g = self._geom
        return [("feature_embedding.weight", g.emb_col, g.dim)]

    def _tail(self, z, rows):
        """No first-order term and no bias: z is not read (None in a group)."""
        W = torch.cat([m.weight for m in self.cross_net_w], dim=0)
        Bv = torch.stack(list(self.cross_net_b), dim=0)
        cn_x = _CrossNet.apply(rows, W, Bv)
        dn_x = self.DN(rows)
        return self.linear(torch.cat([cn_x, dn_x], dim=1))                              # :430-433

    def logit(self, x):
        return self._tail(*self._run(x, True, False))

    def forward(self, x):
        return torch.sigmoid(self.logit(x))                                             # :435


class _AFMAttention(torch.autograd.Function):
    """rows [B, F*D], packed attention parameters -> fc(attention-pooled pair products) [B, 1]: rlctr_afm_fwd / _bwd."""

    @staticmethod
    def forward(ctx, rows, packed, fields, dim, drop_p, rng, masks):
        lib = _lib.load()
        rows, ld = _mlp._rows_view(rows)
        B = rows.shape[0]
        packed = packed.detach().contiguous()
        out = torch.empty(B, 1, dtype=torch.float32, device=rows.device)
        use_rng = drop_p > 0.0 and masks is None
        snap = rng.clone() if use_rng else None                 # the backward regenerates the masks from this snapshot
        _lib.call("rlctr_afm_fwd", lib.rlctr_afm_fwd, rows.data_ptr(), ld, _lib.ptr(packed), _lib.ptr(out), B, fields, dim,
                  float(drop_p), _lib.ptr(snap), _lib.ptr(masks), _lib.stream(), meta={"B": B})
        if use_rng:
            npair = fields * (fields - 1) // 2
            _lib.check(lib.rlctr_rng_advance(_lib.ptr(rng), B * (npair + dim), _lib.stream()), "rlctr_rng_advance")
        ctx.save_for_backward(rows, packed, snap, masks)
        ctx.geom = (ld, fields, dim, float(drop_p))
        return out

    @staticmethod
    def backward(ctx, gout):
        lib = _lib.load()
        rows, packed, snap, masks = ctx.saved_tensors
        ld, fields, dim, drop_p = ctx.geom
        B, fd = rows.shape
        dev = rows.device
        gout = gout.reshape(B).contiguous()
        grows = torch.empty(B, fd, dtype=torch.float32, device=dev)
        dpacked = torch.empty_like(packed)
        ws_bytes = lib.rlctr_afm_ws_bytes(B, dim)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        _lib.call("rlctr_afm_bwd", lib.rlctr_afm_bwd, rows.data_ptr(), ld, _lib.ptr(packed), _lib.ptr(gout), _lib.ptr(grows), fd,
                  _lib.ptr(dpacked), B, fields, dim, drop_p, _lib.ptr(snap), _lib.ptr(masks), _lib.ptr(ws), ws_bytes,
                  _lib.stream(), meta={"B": B})
        return grows, dpacked, None, None, None, None, None


class AFM(_TableModel):
    """p_model.py:438-485  sigma(bias + sum_f w[x_f] + fc(sum_p softmax_p(attention(v_i*v_j)) v_i*v_j)).

    The two ``F.dropout(p=0.2)`` calls of the reference (:477,479) use the default ``training=True``, i.e. they are
    stochastic in ``eval()`` too (SURVEY N6): ``dropout_p`` (0.2) is applied in both modes here as well; set it to 0 for
    a deterministic model.  Masks come from the counter hash of :mod:`.mlp` (own stream; the reference's CPU Philox
    stream is not reproducible on a GPU) or from ``forward(x, masks=[B, P+D])`` in the mask-as-input parity tests."""
    _kind = "fm"
    _fm_term = False

    def __init__(self, feature_nums, field_nums, latent_dims, output_dim=1, device=None):
        super().__init__()
        assert output_dim == 1
        self.feature_nums, self.field_nums, self.latent_dims = feature_nums, int(field_nums), int(latent_dims)
        D = self.latent_dims
        g = Geometry.fm(feature_nums, D)
        self._init_table(g, [(g.emb_col, g.dim)], device)                               # feature_embedding first (:450)
        self.attention_net = nn.Linear(D, D, device=device)                             # :459
        self.attention_softmax = nn.Linear(D, 1, device=device)                         # :462
        self.fc = nn.Linear(D, output_dim, device=device)                               # :465
        with torch.no_grad():                                                           # linear drawn after them (:468)
            dev = self.table.device
            lin = torch.empty(feature_nums, 1, device=dev).normal_() if dev.type == "cuda" else torch.empty(feature_nums, 1).normal_()
            self.table.data[:, g.lin_col:g.lin_col + 1].copy_(lin)
        self.bias = nn.Parameter(torch.zeros((output_dim,), device=device))
        self.dropout_p = 0.2

    def _ref_items(self):
        g = self._geom
        return [("feature_embedding.weight", g.emb_col, g.dim), ("linear.weight", g.lin_col, 1)]

    def _rng_state(self, device):
        st = getattr(self, "_rlctr_rng", None)
        if st is None or st.device != device:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())
            st = torch.tensor([seed, 0], dtype=torch.int64, device=device)
            self._rlctr_rng = st
        return st

    def forward(self, x, masks=None):
        return torch.sigmoid(self.logit(x, masks))

    def logit(self, x, masks=None):
        z, rows = self._run(x, True, False)
        return self._tail(z, rows, masks)

    def _tail(self, z, rows, masks=None):
        """z: bias + first order [B, 1]; the attention term draws its two dropout masks from this model's counter."""
        packed = torch.cat([self.attention_net.weight.reshape(-1), self.attention_net.bias,
                            self.attention_softmax.weight.reshape(-1), self.attention_softmax.bias,
                            self.fc.weight.reshape(-1), self.fc.bias])
        p = float(self.dropout_p)
        rng = self._rng_state(rows.device) if (p > 0.0 and masks is None) else None
        y = _AFMAttention.apply(rows, packed, self.field_nums, self.latent_dims, p, rng, masks)
        return z + y
