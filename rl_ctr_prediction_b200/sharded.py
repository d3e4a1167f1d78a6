"""Row-sharded embedding tables over the GPUs of one box (SURVEY section 8e; BASELINE.json configs[3]).

The reference is single-device; this is how its hot path scales.  One process per GPU (``torch.distributed``, NCCL
over NVLink/NVSwitch).  Samples are data-parallel; every table is row-sharded: ``owner(id) = id mod G``,
``local_row(id) = id div G`` (modulo spreads the Zipf heads of a dictionary-ranked vocabulary); optimizer state
is sharded with the rows.  Dense parameters (bias, tower) are replicated and their gradients all-reduced (NCCL).

Every shard (and every rank's small gradient-side buffers) lives in symmetric memory -- peer-mapped over NVLink -- and
the kernels address it directly:

    forward   rlctr_embed_fwd / rlctr_ffm_fwd read row ``id`` at ``peers[id % G] + (id / G) * pitch``: the gather
              IS the exchange (64 B NVLink reads; measured 529 GB/s for random rows, profiles/r1_symm_probe.md);
    backward  the per-sample rows (dlogit, column sums) are replicated with one ``all_gather``; the source rank PUSHES the
              per-occurrence rows (tower-input gradients) into the owner's receive buffer (posted NVLink writes).  The owner's
              sort / segment-reduce / fused-Adam kernel reads them through ``rlctr_rowgrad.peer_*`` -- local memory, except
              FFM's partner rows, which it reads on the source rank through the peer mapping -- and recomputes the row
              gradient exactly as the single-GPU kernel does.

The ids reach their owners the same way: every rank writes the (local row, global slot) pairs of the ids a peer owns into
that peer's receive buffer and each owner sorts what it received (``shared_sorted_view``; ``RLCTR_SHARD_ROUTE=0``: one
``all_gather`` of the ids and ``rlctr_sort_ids_sharded``).  That sorted view serves the lazy-Adam catch-up and the update.
Two device-side barriers per model step order the phases (catch-up | forward reads ... backward | owner update); nothing
synchronises with the host and no count ever leaves the device, so the sharded step is as graph-capturable as the
single-GPU one.  The owner walks occurrences in (source rank, slot) order: a sharded step is bit-identical from run to
run and equal to the single-GPU step on the concatenated batch.
"""
from __future__ import annotations

import ctypes as C
import os

import torch
import torch.distributed as dist
import torch.nn as nn

from . import _lib
from . import colocated as _co
from . import p_model as Model
from .tables import Geometry, table_struct

# the models with a dense tail (``_tail(z_table, rows)``) besides DeepFM, and the get_model names that differ from the class names
TAIL_KINDS = ("WideAndDeep", "FNN", "InnerPNN", "OuterPNN", "DCN", "AFM")
_ALIASES = {"W&D": "WideAndDeep", "IPNN": "InnerPNN", "OPNN": "OuterPNN"}


def shard_rows(n_rows, world, rank):
    return (n_rows - rank + world - 1) // world if n_rows > rank else 0


def owned_sorted_view_host(ids_all: torch.Tensor, world: int, rank: int, n_rows: int):
    """Host restatement of rlctr_sort_ids_sharded (tests; CPU tensors): (sorted local rows, sorted global slots) of the
    ids this rank owns, in stable (row, position) order -- the owned prefix only, without the sentinel tail."""
    flat = ids_all.reshape(-1).to(torch.int64)
    pos = torch.arange(flat.numel(), dtype=torch.int64)
    mine = (flat >= 0) & (flat < n_rows) & (flat % world == rank)
    rows, pos = flat[mine] // world, pos[mine]
    order = torch.sort(rows, stable=True).indices
    return rows[order], pos[order]


class PeerMemory:
    """One symmetric allocation: the same number of elements on every rank, peer-mapped into every process.
    ``local`` is this rank's tensor, ``ptrs[r]`` the address of rank r's copy in THIS process.  world == 1: a plain
    tensor."""

    def __init__(self, numel, dtype, device, group):
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        if self.world > 1:
            import torch.distributed._symmetric_memory as symm
            self.local = symm.empty(int(numel), dtype=dtype, device=device)
            self.handle = symm.rendezvous(self.local, group if group is not None else dist.group.WORLD)
            self.ptrs = [int(p) for p in self.handle.buffer_ptrs]
        else:
            self.local = torch.empty(int(numel), dtype=dtype, device=device)
            self.handle = None
            self.ptrs = [self.local.data_ptr()]

    def barrier(self):
        """All ranks' work enqueued before this point is complete before any rank's work enqueued after it starts
        (device side, stream ordered: symmetric-memory signal pads, no host involvement)."""
        if self.handle is not None:
            self.handle.barrier(channel=0)


_VIEW_CACHE = {"key": None, "x": None, "view": None}
_ROUTE = {}          # (n, world, device) -> receive buffers of the owner routing


def route_capacity(n, world):
    """Slots each source rank gets in every owner's receive buffer: RLCTR_ROUTE_CAP x the balanced share n / G (default 1.5;
    ids spread by ``id mod G``, so a bucket is Binomial(n, 1/G): 1.5x is > 100 sigma for the uniform benchmark ids, and a
    heavy-hitter id that alone exceeds it trips the overflow flag instead of corrupting the step silently)."""
    f = float(os.environ.get("RLCTR_ROUTE_CAP", "1.5"))
    return ((int(f * n / world) + 1024) + 255) // 256 * 256


def _route_buffers(n, world, dev, group):
    key = (n, world, str(dev))
    rb = _ROUTE.get(key)
    if rb is None:
        cap = route_capacity(n, world)
        keys = PeerMemory(world * cap, torch.int32, dev, group)
        vals = PeerMemory(world * cap, torch.int32, dev, group)
        keys.local.fill_(-1)
        vals.local.zero_()
        rb = {"cap": cap, "keys": keys, "vals": vals, "overflow": torch.zeros(1, dtype=torch.int32, device=dev),
              "kp": (C.c_void_p * 8)(*[int(p) for p in keys.ptrs]), "vp": (C.c_void_p * 8)(*[int(p) for p in vals.ptrs])}
        keys.barrier()
        _ROUTE[key] = rb
    return rb


def check_route_overflow():
    """Host-side check of the routing overflow flags (one device -> host read each; called from flush)."""
    for (n, world, _), rb in _ROUTE.items():
        if int(rb["overflow"].item()) != 0:
            raise _lib.RlctrError(f"owner routing overflow: some rank sent more than {rb['cap']} of its {n} ids to one owner "
                                  f"(skewed ids); the steps since the last check are incomplete.  Rerun with a larger "
                                  f"RLCTR_ROUTE_CAP (now {os.environ.get('RLCTR_ROUTE_CAP', '1.5')}); ShardedCTR models can "
                                  f"also run without routing (RLCTR_SHARD_ROUTE=0), ShardedGroup always routes")


def _route(x, n_rows, group):
    """Owner routing of the batch's ids: every rank writes the (local row, global slot) pairs of the ids a peer owns straight
    into that peer's receive buffer (rlctr_route_ids: posted NVLink writes, a fixed capacity per source), then one device
    barrier.  Returns what the owner's sort of its G * cap received pairs needs: the received ``keys`` (local rows) and
    ``slot_of`` (global slots), ``n_all``, ``n_local``, the sort's outputs ``rows`` and ``out`` (int32 [n_all]) and its
    workspace ``ws`` / ``ws_bytes``; and ``cap`` and ``route_ws`` (the bucket order of this rank's ids, which the routed
    gradient push reuses)."""
    lib = _lib.load()
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    dev, n = x.device, x.numel()
    rb = _route_buffers(n, world, dev, group)
    cap = rb["cap"]
    ws_bytes = lib.rlctr_route_ws_bytes(n, world)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    _lib.call("rlctr_route_ids", lib.rlctr_route_ids, _lib.ptr(x), n, world, rank, n_rows, cap, rb["kp"], rb["vp"],
              _lib.ptr(rb["overflow"]), _lib.ptr(ws), ws_bytes, _lib.stream(), meta={"n": n, "world": world, "cap": cap})
    rb["keys"].barrier()                                         # every source's segment of my receive buffer is complete
    n_all = world * cap
    r = {"keys": rb["keys"].local, "slot_of": rb["vals"].local, "cap": cap, "route_ws": ws, "n_all": n_all,
         "n_local": max(shard_rows(n_rows, world, rank), 1),
         "rows": torch.empty(n_all, dtype=torch.int32, device=dev), "out": torch.empty(n_all, dtype=torch.int32, device=dev)}
    r["ws_bytes"] = lib.rlctr_sort_ws_bytes(n_all, r["n_local"])
    r["ws"] = torch.empty(r["ws_bytes"], dtype=torch.uint8, device=dev)
    return r


def shared_sorted_view(x, n_rows, group):
    """(sorted local rows u32[n_all], sorted global slots u32[n_all], n_all) of the GLOBAL batch as seen by this owner.
    Models that consume the same batch and shard the same vocabulary share it (one exchange + one sort per batch).

    Default (RLCTR_SHARD_ROUTE=1): owner routing -- every rank writes the (local row, global slot) pairs of the ids a peer
    owns straight into that peer's receive buffer (rlctr_route_ids: posted NVLink writes, fixed capacity per source), one
    device barrier, and the owner sorts its G * cap ~ 1.5 n received pairs (rlctr_sort_routed): per-rank work independent
    of G.  RLCTR_SHARD_ROUTE=0: all_gather of the ids + rlctr_sort_ids_sharded over all G * n of them (the first design)."""
    # (the group is not part of the key: models with process groups of their own -- same ranks -- share the view)
    key = (id(x), x._version, x.data_ptr(), tuple(x.shape), int(n_rows))
    if _VIEW_CACHE["key"] == key and _VIEW_CACHE["x"] is x:
        return _VIEW_CACHE["view"]
    lib = _lib.load()
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    dev = x.device
    n = x.numel()
    st = _lib.stream()
    if world > 1 and os.environ.get("RLCTR_SHARD_ROUTE", "1") == "1":
        r = _route(x, n_rows, group)
        _lib.call("rlctr_sort_routed", lib.rlctr_sort_routed, _lib.ptr(r["keys"]), _lib.ptr(r["slot_of"]), r["n_all"], r["n_local"],
                  _lib.ptr(r["rows"]), _lib.ptr(r["out"]), _lib.ptr(r["ws"]), r["ws_bytes"], st, key="rlctr_sort_ids",
                  meta={"n": r["n_all"]})
        view = (r["rows"], r["out"], r["n_all"])
    else:
        ids32 = x.reshape(-1).clamp(-1, n_rows).to(torch.int32)          # out-of-range ids stay out of range in 32 bits
        if world > 1:
            all32 = torch.empty(world * n, dtype=torch.int32, device=dev)
            dist.all_gather_into_tensor(all32, ids32, group=group)
        else:
            all32 = ids32
        n_all = world * n
        srows = torch.empty(n_all, dtype=torch.int32, device=dev)
        sslots = torch.empty(n_all, dtype=torch.int32, device=dev)
        ws_bytes = lib.rlctr_sort_ws_bytes(n_all, n_rows)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        _lib.call("rlctr_sort_ids_sharded", lib.rlctr_sort_ids_sharded, _lib.ptr(all32), n_all, world, rank, n_rows,
                  _lib.ptr(srows), _lib.ptr(sslots), _lib.ptr(ws), ws_bytes, st, key="rlctr_sort_ids", meta={"n": n_all})
        view = (srows, sslots, n_all)
    _VIEW_CACHE.update(key=key, x=x, view=view)
    return view


def routed_view_pos(x, n_rows, group):
    """The routed sorted view with RECEIVE POSITIONS as values (rlctr_sort_routed_pos), plus what the routed gradient push needs:
    {"rows", "pos", "n_all", "cap", "route_ws" (bucket order of this rank's ids), "slot_of" (global slot at every receive position)}."""
    lib = _lib.load()
    r = _route(x, n_rows, group)
    _lib.call("rlctr_sort_routed_pos", lib.rlctr_sort_routed_pos, _lib.ptr(r["keys"]), r["n_all"], r["n_local"], _lib.ptr(r["rows"]),
              _lib.ptr(r["out"]), _lib.ptr(r["ws"]), r["ws_bytes"], _lib.stream(), key="rlctr_sort_ids", meta={"n": r["n_all"]})
    return dict(r, pos=r["out"])


def _dense_member(kind, field_nums, latent_dims, device):
    """The p_model module of ``kind`` as the dense part of a row-sharded model: its bias, tower, cross network or attention and the
    ``_tail`` the stand-alone model runs, without an N-row table of its own (it is built over one row, which is dropped; the owner
    re-homes ``table`` to its shard with :func:`_rehome`)."""
    cls = getattr(Model, kind)
    if kind == "LR":
        m = cls(1, device=device)
    elif kind == "FM":
        m = cls(1, latent_dims, device=device)
    else:
        m = cls(1, field_nums, latent_dims, device=device)
    del m.table
    return m


def _rehome(member, owner, geom):
    """The member reads the owner's shard (not a parameter of the member: the owner lists it once) with geometry ``geom``;
    flush / .to() go through the owner, and the member refuses to train on its own (p_model._TableModel._run)."""
    member.__dict__["table"] = owner.table
    member.__dict__["_group"] = owner
    member._geom = geom
    member._opt, member._stash = None, None


def _copy_dense(dst, src):
    """Every dense parameter of ``src`` (same class as ``dst``) into ``dst``, with what state_dict does not carry: the dropout
    counters (``_rlctr_rng`` of every mlp.Tower and of AFM), AFM's ``dropout_p`` and the train / eval flags."""
    sp = dict(src.named_parameters())
    with torch.no_grad():
        for name, p in dst.named_parameters():
            p.data.copy_(sp[name].data)
    for a, b in zip(dst.modules(), src.modules()):
        a.training = b.training
        st = getattr(b, "_rlctr_rng", None)
        if st is not None:
            a._rlctr_rng = st.clone()
    if hasattr(src, "dropout_p"):
        dst.dropout_p = src.dropout_p


# ---------------------------------------------------------------------------------------------------
class _ShardedTable(nn.Module):
    """What ShardedCTR and ShardedGroup share: the process group, this rank's shard of the table in symmetric memory (the
    ``table`` Parameter, which optim.Adam hands back to this module), the device barrier, the table structs the kernels see, the
    lazy-Adam catch-up of the owned rows and the all-reduce of the dense gradients.  Every rank must call the same methods in the
    same order (they contain device barriers)."""

    def __init__(self, feature_nums, group, device):
        super().__init__()
        self.feature_nums, self.group = int(feature_nums), group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        if self.world not in (1, 2, 4, 8):
            raise _lib.RlctrError("row sharding supports 1, 2, 4 or 8 GPUs (owner = id & (G-1))")
        self._n_local = max(shard_rows(self.feature_nums, self.world, self.rank), 1)
        self._dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self._opt, self._stash, self._ws = None, None, {}
        # True when `group` is used by this model alone: its step may then run as a parallel branch of a captured graph
        # (graphs.GraphedTrainStep), overlapping its NVLink-bound gathers with another model's GEMMs
        self.fork_ok = False

    def _alloc_table(self, col_groups):
        """The shard [n_alloc, row_pitch] (the same allocation on every rank) as the ``table`` Parameter: zeros, and N(0, 1) in
        every list of columns of ``col_groups`` (one draw per list) over the owned rows."""
        n_alloc, pitch = max(shard_rows(self.feature_nums, self.world, 0), 1), self._geom.row_pitch
        self._pm = PeerMemory(n_alloc * pitch, torch.float32, self._dev, self.group)
        data = self._pm.local.view(n_alloc, pitch)
        data.zero_()
        for cols in col_groups:
            data[:self._n_local, cols] = torch.randn(self._n_local, len(cols), device=self._dev)
        self.table = nn.Parameter(data)
        self.table._rlctr_owner = self

    def _copy_shard(self, full):
        """This rank's rows (ids rank, rank + G, ...) of a single-GPU table [N, row_pitch] into the shard."""
        with torch.no_grad():
            shard = full[self.rank::self.world]
            self.table.data[:shard.shape[0]].copy_(shard)

    # ---- protocol shared with optim.Adam / graphs ----------------------------------------------------------------------
    def _apply(self, fn, recurse=True):
        saved = self._parameters.pop("table")            # the shard lives in symmetric memory: .to()/.cuda() must not move it
        out = super()._apply(fn, recurse)
        self._parameters["table"] = saved
        self.table._rlctr_owner = self
        return out

    def flush(self):
        if self._opt is not None:
            self._opt.flush(self.table.data)
        check_route_overflow()

    def zero_grad(self, set_to_none=True):
        self._stash = None
        return super().zero_grad(set_to_none)

    def barrier(self):
        self._pm.barrier()

    _reduce_ws = Model._TableModel._reduce_ws
    _rows_ws = Model._TableModel._rows_ws

    def gather_table(self):
        """The full table [N, row_pitch], rebuilt on every rank (tests / checkpointing)."""
        self.flush()
        mine = self.table.data.contiguous()
        if self.world == 1:
            return mine[:self.feature_nums].clone()
        parts = [torch.empty_like(mine) for _ in range(self.world)]
        dist.all_gather(parts, mine, group=self.group)
        full = torch.empty(self.feature_nums, self._geom.row_pitch, dtype=torch.float32, device=mine.device)
        for r in range(self.world):
            full[r::self.world] = parts[r][:shard_rows(self.feature_nums, self.world, r)]
        return full

    def _local_struct(self):
        """The shard as the optimizer kernels see it: n_local rows, local row ids."""
        return table_struct(self.table.data, self._geom)

    def _global_struct(self):
        """The whole table as the forward gathers see it: global ids, peers[] = every rank's shard."""
        g = self._geom
        t = _lib.Table(self.table.data.data_ptr(), self.feature_nums, g.row_stride, g.lin_col, g.emb_col, g.dim, g.row_pitch)
        if self.world > 1:
            t.world = self.world
            for r, p in enumerate(self._pm.ptrs):
                t.peers[r] = p
        return t

    # ---- pieces of the step -------------------------------------------------------------------------------------------
    def _catchup(self, srows, n_all, F, key):
        """Lazy Adam: bring the owned rows of the sorted view up to date before any rank reads them."""
        opt = self._opt
        if opt is not None and opt.lazy and opt.dirty:
            lib = _lib.load()
            t, a = self._local_struct(), opt.struct()
            _lib.call("rlctr_rows_catchup", lib.rlctr_rows_catchup, _lib.ptr(srows), n_all, C.byref(t), C.byref(a), _lib.stream(),
                      key=key, meta=self._meta(n_all // F, F))

    def _allreduce_dense(self):
        """Sum every dense gradient over the ranks: one all_reduce of them all, flattened."""
        dense = [p for p in self.parameters() if p is not self.table and p.grad is not None]
        flat = torch.cat([p.grad.reshape(-1) for p in dense])
        dist.all_reduce(flat, group=self.group)
        o = 0
        for p in dense:
            p.grad = flat[o:o + p.numel()].view_as(p).clone()
            o += p.numel()


class ShardedCTR(_ShardedTable):
    """LR / FM / FFM / DeepFM, and the tail models WideAndDeep / FNN / InnerPNN / OuterPNN / DCN / AFM, with the table row-sharded
    over the process group.  A tail model keeps its stand-alone row (16 floats, with or without the first-order column); its dense
    part is the p_model module itself (``dense``: bias, tower, cross network or attention, and its ``_tail``).

    ``train_step(features, labels, optimizer)`` is the reference loop body (src/main/pretrain_main.py:96-102) for
    the local batch; ``forward(features)`` is the frozen scoring pass.  ``from_model`` shards an existing
    single-GPU model (for the 1-vs-G equivalence check); ``gather_table`` rebuilds the full fused table on every
    rank.  Every rank must call the same methods in the same order (they contain device barriers).

    The owners get the gradient side of remote samples by PUSH: the per-sample rows (dlogit, or the sums rows that carry it)
    are replicated with one all_gather, and the source ranks WRITE the per-occurrence rows (the tower-input gradients) into the
    owners' memory, so the update reads local memory only -- but for FFM's 600-byte partner rows, which it reads on the source
    rank through the peer mapping."""

    def __init__(self, kind, feature_nums, field_nums, latent_dims, group=None, device=None):
        kind = _ALIASES.get(kind, kind)
        if kind not in ("LR", "FM", "FFM", "DeepFM") + TAIL_KINDS:
            raise _lib.RlctrError(f"ShardedCTR: unknown model {kind!r} (LR, FM, FFM, DeepFM, {', '.join(TAIL_KINDS)})")
        super().__init__(feature_nums, group, device)
        self.kind, self.field_nums, self.latent_dims = kind, int(field_nums), int(latent_dims)
        if kind == "LR":
            g = Geometry.lr(self._n_local)
        elif kind == "FFM":
            g = Geometry.ffm(self._n_local, self.field_nums, self.latent_dims)
        else:
            g = Geometry.fm(self._n_local, self.latent_dims, with_linear=kind not in ("FNN", "InnerPNN", "OuterPNN", "DCN"))
        self._geom = g = g.with_state()
        self._kind = {"LR": "lr", "FFM": "ffm"}.get(kind, "fm")
        self._fm_term = kind in ("FM", "DeepFM")
        self._alloc_table([([g.lin_col] if g.lin_col >= 0 else []) + list(range(g.emb_col, g.emb_col + g.dim))])
        self.dense = None
        if kind in TAIL_KINDS:
            self.dense = _dense_member(kind, self.field_nums, self.latent_dims, self._dev)
            _rehome(self.dense, self, g)
            self.bias = getattr(self.dense, "bias", None)         # W&D, AFM: the member's own bias; FNN, PNN, DCN: none
        else:
            self.bias = nn.Parameter(torch.zeros(1, device=self._dev))
        self.mlp = Model._tower(self.field_nums * self.latent_dims, self._dev) if kind == "DeepFM" else None
        self._gbuf, self._xbuf = {}, {}
        self._after_gather = None

    def _meta(self, B, F):
        g = self._geom
        return {"model": "Sharded" + self.kind, "B": B, "F": max(F, 1), "rs": g.row_stride, "dim": g.dim, "n_rows": g.n_rows,
                "lin": g.lin_col >= 0}

    @property
    def _has_tail(self):
        return self.mlp is not None or self.dense is not None

    def _tail(self, z, rows):
        """Logit [B, 1] from the table part z [B, 1] and the gathered rows [B, F*D]: the stand-alone model's ``_tail``."""
        if self.dense is not None:
            return self.dense._tail(z, rows)
        return z + self.mlp(rows)                             # DeepFM

    @classmethod
    def from_model(cls, model, group=None):
        """Shard a single-GPU p_model instance (same parameters on every rank) over the group: its table, its dense parameters,
        and the dropout counters and train / eval flags of its tower, cross network or attention."""
        kind = type(model).__name__
        self = cls(kind, model.feature_nums, getattr(model, "field_nums", 15), getattr(model, "latent_dims", 1),
                   group=group, device=model.table.device)
        self._copy_shard(model.table.data)
        if self.dense is not None:
            _copy_dense(self.dense, model)                   # bias (W&D, AFM), towers, cross network, attention
        else:
            with torch.no_grad():
                self.bias.data.copy_(model.bias.data)
            if self.mlp is not None:
                _copy_dense(self.mlp, model.mlp)             # DeepFM's tower
        self.barrier()
        return self

    def _grad_buffers(self, B, F):
        """dlogit [B] | sums [B, rs] | extra [B, F*D] | staged [B*F, rs] in ONE symmetric allocation per batch size: this rank's
        gradient side of the step (the owners read the staged FFM partner rows in place, through ``staged_ptrs``)."""
        buf = self._gbuf.get(B)
        if buf is not None:
            return buf
        g = self._geom
        sizes = {"dlogit": (B + 3) // 4 * 4,
                 "sums": B * g.row_stride if self._fm_term else 0,
                 "extra": B * F * g.dim if self._has_tail else 0,
                 "staged": B * F * g.row_stride if self._kind == "ffm" else 0}
        total = sum(sizes.values())
        pm = PeerMemory(total, torch.float32, self.table.device, self.group)
        buf, off = {"pm": pm}, 0
        for k, sz in sizes.items():
            if sz:
                buf[k] = pm.local[off:off + sz]
                buf[k + "_ptrs"] = [p + 4 * off for p in pm.ptrs]
            else:
                buf[k], buf[k + "_ptrs"] = None, None
            off += sz
        self._gbuf[B] = buf
        return buf

    def _exchange_buffers(self, B, F):
        """Receive side of the push for batch size B: the all-gathered per-sample rows of every rank (plain local tensors) and
        the symmetric buffer the sources write the per-occurrence tail gradients into."""
        xb = self._xbuf.get(B)
        if xb is not None:
            return xb
        g, dev, G = self._geom, self.table.device, self.world
        bp = (B + 3) // 4 * 4
        xb = {"dlogit_all": torch.empty(G * bp, dtype=torch.float32, device=dev), "bp": bp, "sums_all": None, "recv": None}
        if self._fm_term:
            xb["sums_all"] = torch.empty(G * B * g.row_stride, dtype=torch.float32, device=dev)
        if self._has_tail:
            pm = PeerMemory(G * B * F * g.dim, torch.float32, dev, self.group)
            pm.local.zero_()
            xb["recv"] = pm
            xb["recv_ptrs"] = (C.c_void_p * 8)(*[int(p) for p in pm.ptrs])
        self._xbuf[B] = xb
        return xb

    # ---- the step ---------------------------------------------------------------------------------
    def _interact(self, x, buf, train):
        """The single-GPU interaction kernels reading rows through the peer table.  Returns (logit[B], tower rows)."""
        lib = _lib.load()
        B, F = x.shape
        dev = x.device
        g = self._geom
        t = self._global_struct()
        logit = torch.empty(B, dtype=torch.float32, device=dev)
        trows = None
        if self._kind == "ffm":
            partners = buf["staged"] if train else None
            _lib.call("rlctr_ffm_fwd", lib.rlctr_ffm_fwd, _lib.ptr(x), C.byref(t), _lib.ptr(self.bias.data), _lib.ptr(logit),
                      None, 1, _lib.ptr(partners), B, F, self.latent_dims, _lib.stream(), key="rlctr_ffm_fwd[sharded]",
                      meta=self._meta(B, F))
        else:
            sums = buf["sums"] if (train and self._fm_term) else None
            pitch = 0
            if self._has_tail:
                pitch = (F * g.dim + 3) // 4 * 4
                trows = torch.empty(B, pitch, dtype=torch.float32, device=dev)
            flags = _lib.RLCTR_FM_TERM if self._fm_term else 0
            bias = self.bias.data if self.bias is not None else None
            _lib.call("rlctr_embed_fwd", lib.rlctr_embed_fwd, _lib.ptr(x), C.byref(t), _lib.ptr(bias), _lib.ptr(logit),
                      None, 1, _lib.ptr(sums), _lib.ptr(trows), pitch, B, F, flags, _lib.stream(),
                      key=f"rlctr_embed_fwd[Sharded{self.kind}]",
                      meta=dict(self._meta(B, F), sums=sums is not None, rows=trows is not None, n_rows=self.feature_nums))
            if trows is not None and pitch != F * g.dim:
                trows = trows[:, :F * g.dim]
        return logit, trows

    @torch.no_grad()
    def forward(self, x):
        x = Model._check_ids(x)
        self.flush()
        self.barrier()                                        # every shard is settled before anyone reads it
        logit, trows = self._interact(x, None, train=False)
        if self._has_tail:
            logit = self._tail(logit.view(-1, 1), trows).reshape(-1)
        self.barrier()                                        # nobody starts writing rows while a peer still reads
        return torch.sigmoid(logit).reshape(-1, 1)

    def train_step(self, features, labels, optimizer):
        """One step on the local batch; the update equals the single-GPU step on the concatenated global
        batch.  Returns the local mean BCE loss (device scalar)."""
        lib = _lib.load()
        x = Model._check_ids(features)
        B, F = x.shape
        G, st = self.world, _lib.stream()
        y = _co.labels(labels)
        buf = self._grad_buffers(B, F)
        srows, sslots, n_all = shared_sorted_view(x, self.feature_nums, self.group)
        self._catchup(srows, n_all, F, f"rlctr_rows_catchup[Sharded{self.kind}]")
        self.barrier()                                        # B1: all owners caught their rows up | forward reads
        logit, trows = self._interact(x, buf, train=True)
        hook, self._after_gather = self._after_gather, None     # graphs.GraphedTrainStep: fork point of the captured step
        if hook is not None:
            hook()
        loss = torch.empty(1, dtype=torch.float32, device=x.device)
        for p in self.parameters():
            p.grad = None
        dlogit, grad = _co.loss_head(self, logit, trows, y, loss.data_ptr(), self._reduce_ws(x.device), dl=buf["dlogit"][:B],
                                     scale=1.0 / G)
        if grad is not None:
            buf["extra"].view(B, -1).copy_(grad)
        dz_in_sums = G > 1 and self._fm_term
        if dz_in_sums:                                        # one aligned 64 B line per occurrence for the owners to read
            buf["sums"].view(B, -1)[:, -1] = dlogit
        peer = None
        if G > 1:
            self._allreduce_dense()
            xb, g = self._exchange_buffers(B, F), self._geom
            peer = {"world": G, "n_per_rank": B * F, "staged": buf["staged_ptrs"], "sums": None, "extra": None,
                    "dlogit": [xb["dlogit_all"].data_ptr() + r * 4 * xb["bp"] for r in range(G)]}    # not read with dz_in_sums
            if dz_in_sums:                                    # dlogit rides in the sums rows: one all_gather serves both
                dist.all_gather_into_tensor(xb["sums_all"], buf["sums"], group=self.group)
                peer["sums"] = [xb["sums_all"].data_ptr() + r * 4 * B * g.row_stride for r in range(G)]
            else:
                dist.all_gather_into_tensor(xb["dlogit_all"], buf["dlogit"], group=self.group)
            if xb["recv"] is not None:                        # per-occurrence rows: posted writes into the owners' memory
                n = B * F
                _lib.call("rlctr_push_rows", lib.rlctr_push_rows, _lib.ptr(x), n, G, self.rank, self.feature_nums,
                          _lib.ptr(buf["extra"]), g.dim, xb["recv_ptrs"], st, meta={"n": n, "width": g.dim})
                peer["extra"] = [xb["recv"].local.data_ptr() + r * 4 * n * g.dim for r in range(G)]
        self.barrier()                                        # B2: every rank's gradient-side buffers are complete
        self._stash = Model.RowsStash(sorted_ids=srows, sorted_slots=sslots, n=n_all, dlogit=dlogit, sums=buf["sums"],
                                      extra=buf["extra"], staged=buf["staged"], fields=F,
                                      flags=(_lib.RLCTR_STAGED_PARTNER if buf["staged"] is not None else 0) |
                                            (_lib.RLCTR_DZ_IN_SUMS if dz_in_sums else 0), peer=peer)
        optimizer.step()
        return loss.reshape(())


# ---------------------------------------------------------------------------------------------------
class ShardedGroup(_co._GroupStep, _ShardedTable):
    """Co-located records (colocated.py) over a row-sharded joint table: the members ``colocate()`` accepts (LR, FM, DeepFM,
    WideAndDeep, FNN, InnerPNN, OuterPNN, DCN, AFM) trained on the same id stream share one 384-byte record per id,
    ``owner(id) = id mod G``.  Per step and rank: ONE routed sorted view (shared_sorted_view), one catch-up of the owned records, one
    gather through the peer mapping (rlctr_group_fwd: one NVLink read per (sample, field) for all members instead of one per
    member), one all_gather of the per-sample rows [B, 32] = column sums + the dL/dlogit of every member with a first-order or FM
    column, ONE push of every dense-tail member's per-occurrence gradients (rlctr_push_rows_routed_multi: one interleaved row per
    occurrence), one all_reduce of all dense gradients, two device barriers, one update (rlctr_group_rows_adam).  The update equals
    the single-GPU group step on the concatenated global batch.  ``members[i]`` is the member's p_model module without a table of
    its own: its bias, tower, cross network or attention, and the ``_tail`` the group step runs."""

    SUMS_PITCH = 32                    # floats per sample of the exchange row: S | dL/dlogit of members 0..3 in the last four columns.
                                       # One line (S <= 28 floats); with max_lines > 1 the instance widens it to the whole lines
                                       # that hold rs + 4 floats
    _UPDATE_KEY = "rlctr_group_rows_adam[ShardedGroup]"

    def __init__(self, kinds, feature_nums, field_nums, latent_dims, group=None, device=None, max_lines=1):
        kinds = tuple(_ALIASES.get(k, k) for k in kinds)
        names = tuple(c.__name__ for c in _co.MEMBER_KINDS)
        if not all(k in names for k in kinds) or not 1 <= len(kinds) <= _lib.RLCTR_GROUP_MAX:
            raise _lib.RlctrError(f"ShardedGroup members: {', '.join(names)} (up to {_lib.RLCTR_GROUP_MAX}); got {', '.join(kinds)}")
        super().__init__(feature_nums, group, device)
        self.kinds, self.field_nums, self.latent_dims = kinds, int(field_nums), int(latent_dims)
        members = [_dense_member(k, self.field_nums, self.latent_dims, self._dev) for k in kinds]
        self._cols, used = _co._layout(members, max_lines)
        rs = (used + 1 + 3) // 4 * 4
        if max_lines == 1 and rs > self.SUMS_PITCH - _lib.RLCTR_GROUP_MAX:
            raise _lib.RlctrError("joint row too wide for the per-sample exchange row (28 floats); pass max_lines=2 for a "
                                  "two-line exchange row")
        if max_lines > 1:
            self.SUMS_PITCH = (rs + _lib.RLCTR_GROUP_MAX + 31) // 32 * 32
        self._geom = _co._record(self._n_local, used)
        self._max_lines = max_lines
        self._alloc_table([([lin] if lin >= 0 else []) + list(range(emb, emb + dim)) for lin, emb, dim in self._cols])
        wide = _co._wide(members, used)
        for m, col in zip(members, self._cols):
            _rehome(m, self, _co._member_view(m, self._geom, col, wide))
        self.members = nn.ModuleList(members)
        self._buf = {}

    @property
    def biases(self):
        """The members' bias parameters (None for FNN, InnerPNN, OuterPNN, DCN)."""
        return [getattr(m, "bias", None) for m in self.members]

    @property
    def mlps(self):
        """The members' towers (``mlp``; nn.Identity for a member without one)."""
        return [m.mlp if getattr(m, "mlp", None) is not None else nn.Identity() for m in self.members]

    def _meta(self, B, F):
        g = self._geom
        return {"model": "Sharded" + "+".join(self.kinds), "B": B, "F": max(F, 1), "rs": g.row_stride, "dim": g.dim,
                "n_rows": g.n_rows, "lin": False, "members": [(k, c[2]) for k, c in zip(self.kinds, self._cols)]}

    @classmethod
    def from_group(cls, cg, group=None):
        """Shard a single-GPU colocated.ColocatedCTR (same parameters on every rank) over the process group: the joint table, every
        member's dense state and its dropout counters."""
        kinds = [type(m).__name__ for m in cg.members]
        F = next((m.field_nums for m in cg.members if hasattr(m, "field_nums")), 15)
        self = cls(kinds, cg.feature_nums, F, max(getattr(m, "latent_dims", 1) for m in cg.members),
                   group=group, device=cg.table.device, max_lines=cg._max_lines)
        assert self._cols == cg._cols
        cg.flush()
        self._copy_shard(cg.table.data)
        for dst, src in zip(self.members, cg.members):
            _copy_dense(dst, src)
        self.barrier()
        return self

    def _tail_sources(self):
        """[(member, float offset in the interleaved receive row, width)] of the members with a dense tail, and the row's pitch:
        each member's dim rounded up to even (the push moves 8-byte pieces)."""
        out, off = [], 0
        for i, m in enumerate(self.members):
            if hasattr(m, "_tail"):
                w = (self._cols[i][2] + 1) // 2 * 2
                out.append((i, off, w))
                off += w
        return out, off

    def _uses_dz(self, i):
        """Member i reads its dL/dlogit in the update (a first-order column or the FM term); a tail-only member does not."""
        lin, _, dim = self._cols[i]
        return lin >= 0 or (self.members[i]._fm_term and dim > 0)

    def _exchange(self, B, F):
        """Per batch size: this rank's per-sample exchange rows [B, 32], their all-gathered copy [G*B, 32], and the ONE symmetric
        receive buffer [G * cap, pitch] the source ranks push every dense-tail member's per-occurrence gradients into."""
        b = self._buf.get(B)
        if b is None:
            dev, G = self.table.device, self.world
            b = {"sums": torch.zeros(B, self.SUMS_PITCH, dtype=torch.float32, device=dev),
                 "sums_all": torch.zeros(G * B, self.SUMS_PITCH, dtype=torch.float32, device=dev), "recv": None}
            srcs, pitch = self._tail_sources()
            if srcs and G > 1:                                # dense per-source segments of interleaved rows (routed push)
                pm = PeerMemory(G * route_capacity(B * F, G) * pitch, torch.float32, dev, self.group)
                pm.local.zero_()
                b["recv"] = (pm, (C.c_void_p * 8)(*[int(p) for p in pm.ptrs]))
            self._buf[B] = b
        return b

    @torch.no_grad()
    def forward(self, x):
        """pCTR of every member, float32 [B, M] (as colocated.ColocatedCTR.forward, the rows read through the peer mapping)."""
        x = Model._check_ids(x)
        self.flush()
        self.barrier()                                        # every shard is settled before anyone reads it
        out = self._pctr(x, "rlctr_group_fwd[sharded infer]")
        self.barrier()                                        # nobody starts writing rows while a peer still reads
        return out

    def train_step(self, features, labels, optimizer):
        """One step of every member on the local batch; returns the local mean BCE losses, float32 [M]."""
        lib = _lib.load()
        if self._opt is None:
            raise _lib.RlctrError("build rl_ctr_prediction_b200.optim.Adam(group.parameters(), ...) before training the group")
        x = Model._check_ids(features)
        B, F = x.shape
        st, G, M = _lib.stream(), self.world, len(self.members)
        y = _co.labels(labels)
        buf = self._exchange(B, F)
        view = None
        if G > 1:                                             # routed exchange: positions in the owner's receive buffers
            view = routed_view_pos(x, self.feature_nums, self.group)
            srows, sslots, n_all = view["rows"], view["pos"], view["n_all"]
        else:
            srows, sslots, n_all = shared_sorted_view(x, self.feature_nums, self.group)
        self._catchup(srows, n_all, F, "rlctr_rows_catchup[ShardedGroup]")
        self.barrier()                                        # B1: all owners caught their rows up | forward reads
        arr, logits, rows = self._member_structs(B, F, x.device, True)
        t = self._global_struct()
        sums = buf["sums"]
        _lib.call("rlctr_group_fwd", lib.rlctr_group_fwd, _lib.ptr(x), C.byref(t), arr, M, _lib.ptr(sums), self.SUMS_PITCH, B, F, st,
                  key="rlctr_group_fwd[ShardedGroup]", meta=dict(self._meta(B, F), n_rows=self.feature_nums))
        losses, dlogits, extras = self._heads(F, logits, rows, y, scale=1.0 / G)
        for i, dl in enumerate(dlogits):
            if self._uses_dz(i):
                sums[:, self.SUMS_PITCH - _lib.RLCTR_GROUP_MAX + i] = dl    # dL/dlogit rides in the sample's exchange row
        pitches = [0] * M
        if G > 1:
            self._allreduce_dense()
            dist.all_gather_into_tensor(buf["sums_all"], sums, group=self.group)
            sums = buf["sums_all"]
            if buf["recv"] is not None:                       # ONE push of every tail member's per-occurrence rows, in the routed
                pm, ptrs = buf["recv"]                        # bucket order: interleaved rows, coalesced posted writes
                n = B * F
                tails, pitch = self._tail_sources()
                keep = []
                for i, off, w in tails:
                    src = extras[i].view(n, -1)
                    if src.shape[1] != w:                     # odd dim: a zero pad column (carried, never read by the update)
                        src = torch.nn.functional.pad(src, (0, w - src.shape[1]))
                    keep.append(src)
                srcs = (C.c_void_p * len(keep))(*[s_.data_ptr() for s_ in keep])
                widths = (C.c_int32 * len(keep))(*[w for _, _, w in tails])
                _lib.call("rlctr_push_rows_routed_multi", lib.rlctr_push_rows_routed_multi, _lib.ptr(view["route_ws"]), n, G,
                          self.rank, view["cap"], srcs, widths, len(keep), ptrs, st, key="rlctr_push_rows",
                          meta={"n": n, "width": pitch, "sources": len(keep)})
                for i, off, _ in tails:
                    extras[i], pitches[i] = pm.local[off:], pitch
        self.barrier()                                        # B2: every rank's gradient-side buffers are complete
        self._stash = _co.GroupStash(sorted_ids=srows, sorted_slots=sslots, n=n_all, fields=F, sums=sums, dlogit=[None] * M,
                                     extra=extras, sums_pitch=self.SUMS_PITCH, world=G, extra_pitch=pitches,
                                     slot_of=view["slot_of"] if view is not None else None)
        optimizer.step()
        return losses
