"""Row-sharded training of the tower-tail models (rl_ctr_prediction_b200/sharded.py): ShardedGroup takes every member colocate()
takes, ShardedCTR the six tail models stand-alone, and the dense-tail gradients of all of a group's members travel in ONE routed
push (rlctr_push_rows_routed_multi) as interleaved receive rows that the update reads with rlctr_member.extra_pitch.

World 1 runs a real one-rank NCCL group; G = 2, 4, 8 ranks are emulated on one GPU at the kernel level (the receive buffers of all
owners live in one device memory), as tests/test_gpu_kernels.py::test_owner_routing_equals_gather_and_sort does.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import state_from_golden
from test_gpu_colocated_tails import COMBOS, NAMES, _rng_counters, _set_dropout

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
F, D = 15, 10


@pytest.fixture(scope="module")
def one_rank():
    import torch.distributed as dist
    if not dist.is_initialized():
        import socket
        s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
        dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=0, world_size=1,
                                device_id=torch.device(DEV))
    yield None
    if dist.is_initialized():
        dist.destroy_process_group()


def _models(names, N, seed, dropout):
    from rl_ctr_prediction_b200 import pretrain_main as PM
    torch.manual_seed(seed)
    ms = [PM.get_model(NAMES[n], N, F, D).to(DEV).train() for n in names]
    for i, m in enumerate(ms):
        _set_dropout(m, dropout, 1000 * seed + 10 * i)
    return ms


def _batches(N, B, steps, seed, zipf=False):
    g = torch.Generator().manual_seed(seed)
    per = N // F
    out = []
    for _ in range(steps):
        if zipf:
            x = (torch.rand(B, F, generator=g) ** 6 * per).long().clamp_(0, per - 1)
        else:
            x = torch.randint(0, per, (B, F), generator=g)
        x = x + torch.arange(F) * per
        y = (torch.rand(B, generator=g) < 0.3).long()
        out.append((x.to(DEV), y.to(DEV)))
    return out


def _dense_params(m):
    return {k: p for k, p in m.named_parameters() if k != "table"}


def _assert_group_state_equal(sg, cg):
    cg.flush()
    assert torch.equal(sg.gather_table(), cg.table.data)
    for a, b in zip(sg.members, cg.members):
        pa, pb = _dense_params(a), _dense_params(b)
        assert set(pa) == set(pb)
        for k in pb:
            assert torch.equal(pa[k], pb[k]), (type(b).__name__, k)
        assert _rng_counters(a) == _rng_counters(b), type(b).__name__


# ---- 1. world 1: ShardedGroup.from_group(cg) == ColocatedCTR, bit for bit --------------------------------------------------------
@pytest.mark.parametrize("mode", ["lazy", "dense"])
@pytest.mark.parametrize("zipf", [False, True])
@pytest.mark.parametrize("names", COMBOS)
def test_world1_group_equals_colocated(one_rank, names, zipf, mode):
    from rl_ctr_prediction_b200 import colocated, optim, sharded
    N, B, steps = 3001, 384, 4
    cg = colocated.colocate(_models(names, N, seed=21, dropout=False))
    sg = sharded.ShardedGroup.from_group(cg)
    oa = optim.Adam(cg.parameters(), lr=1e-3, weight_decay=1e-5, mode=mode)
    ob = optim.Adam(sg.parameters(), lr=1e-3, weight_decay=1e-5, mode=mode)
    for x, y in _batches(N, B, steps, seed=6, zipf=zipf):
        assert torch.equal(cg.train_step(x, y, oa), sg.train_step(x, y, ob))
    _assert_group_state_equal(sg, cg)
    x = _batches(N, B, 1, seed=8)[0][0]
    assert torch.equal(sg(x), cg(x))


@pytest.mark.parametrize("names", COMBOS)
def test_world1_group_equals_colocated_dropout_on(one_rank, names):
    """Towers in train(), AFM's attention dropout at 0.2: from_group copies the dropout counters, so both draw the same masks."""
    from rl_ctr_prediction_b200 import colocated, optim, sharded
    N, B, steps = 2500, 256, 4
    cg = colocated.colocate(_models(names, N, seed=7, dropout=True))
    sg = sharded.ShardedGroup.from_group(cg)
    oa = optim.Adam(cg.parameters(), lr=1e-3, weight_decay=1e-5)
    ob = optim.Adam(sg.parameters(), lr=1e-3, weight_decay=1e-5)
    for x, y in _batches(N, B, steps, seed=5):
        assert torch.equal(cg.train_step(x, y, oa), sg.train_step(x, y, ob))
    _assert_group_state_equal(sg, cg)
    for m, n in zip(cg.members, names):
        if n not in ("LR", "FM"):
            assert all(c > 0 for c in _rng_counters(m)), n                 # the masks were drawn
    x = _batches(N, B, 1, seed=9)[0][0]
    assert torch.equal(sg(x), cg(x))
    _assert_group_state_equal(sg, cg)


# ---- 2. built from kinds: no stand-alone tables, every dense parameter listed once ------------------------------------------------
@pytest.mark.parametrize("kinds", [("AFM", "LR", "DCN"), ("DeepFM", "IPNN"), ("W&D", "OPNN")])     # get_model names
def test_group_from_kinds_trains_without_member_tables(one_rank, kinds):
    from rl_ctr_prediction_b200 import optim, pretrain_main as PM, sharded
    N, B = 20011, 256
    sg = sharded.ShardedGroup(kinds, N, F, D)
    ref = [PM.get_model(k, 7, F, D) for k in kinds]
    dense = sum(p.numel() for m in ref for n_, p in m.named_parameters() if n_ != "table")
    params = list(sg.parameters())
    assert len({id(p) for p in params}) == len(params)
    assert sum(p.numel() for p in params) == sg.table.numel() + dense
    assert all(p is sg.table or p.shape[0] < N for p in params)
    opt = optim.Adam(sg.parameters(), lr=1e-3, weight_decay=1e-5)
    member_params = {id(p) for m in sg.members for p in m.parameters()}
    assert member_params == {id(p) for p in opt._dense}
    before = {k: p.detach().clone() for k, p in sg.named_parameters() if p is not sg.table}
    for x, y in _batches(N, B, 3, seed=3):
        losses = sg.train_step(x, y, opt)
        assert bool(torch.isfinite(losses).all())
    for k, p in sg.named_parameters():
        if p is not sg.table:
            assert not torch.equal(before[k], p.detach()), k
    assert sg(_batches(N, B, 1, seed=4)[0][0]).shape == (B, len(kinds))


# ---- 3. ShardedCTR for the six tail models: the reference's golden trajectory ----------------------------------------------------
@pytest.mark.parametrize("name", ["WideAndDeep", "FNN", "InnerPNN", "OuterPNN", "DCN", "AFM"])
def test_sharded_tail_world1_matches_reference(golden, golden_tails, name, one_rank):
    from test_gpu_models import assert_state, build, close, load
    from rl_ctr_prediction_b200 import optim, sharded
    single = load(build(NAMES[name], 255), state_from_golden(golden_tails, f"train/{name}/init")).to(DEV)
    if name == "AFM":
        single.dropout_p = 0.0
    m = sharded.ShardedCTR.from_model(single)
    m.eval()                                               # dropout off, as in the golden trajectories
    assert m.mlp is None and (m.bias is not None) == (name in ("WideAndDeep", "AFM"))
    opt = optim.Adam(params=m.parameters(), lr=1e-3, weight_decay=1e-5)
    for s in range(3):
        x = torch.as_tensor(golden["train/x"][s]).to(DEV)
        y = torch.as_tensor(golden["train/y"][s]).to(DEV)
        with torch.no_grad():
            close(m(x), golden_tails[f"train/{name}/pctr{s}"])
        close(m.train_step(x, y, opt), golden_tails[f"train/{name}/loss{s}"])
    full = m.gather_table()
    single.table.data.copy_(full)
    sp = dict(single.named_parameters())
    with torch.no_grad():
        for k, p in m.dense.named_parameters():
            sp[k].data.copy_(p)
    assert_state(single, state_from_golden(golden_tails, f"train/{name}/final"))


# ---- 4. G ranks emulated on one GPU ------------------------------------------------------------------------------------------------
def _ptr(t):
    return t.data_ptr() if t is not None else None


def _route(lib, ids, world, N, cap):
    """Every emulated source rank routes its ids: (receive keys / vals of every owner, each source's routing workspace)."""
    from rl_ctr_prediction_b200 import _lib
    n = ids.shape[1]
    keys = [torch.full((world * cap,), -1, dtype=torch.int32, device=DEV) for _ in range(world)]
    vals = [torch.zeros(world * cap, dtype=torch.int32, device=DEV) for _ in range(world)]
    kp = (C.c_void_p * 8)(*[k.data_ptr() for k in keys])
    vp = (C.c_void_p * 8)(*[v.data_ptr() for v in vals])
    flag = torch.zeros(1, dtype=torch.int32, device=DEV)
    wsb = lib.rlctr_route_ws_bytes(n, world)
    wss = []
    for r in range(world):
        ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
        _lib.check(lib.rlctr_route_ids(_ptr(ids[r]), n, world, r, N, cap, kp, vp, _ptr(flag), _ptr(ws), wsb, _lib.stream()),
                   "rlctr_route_ids")
        wss.append(ws)
    assert int(flag.item()) == 0
    return keys, vals, wss


@pytest.mark.parametrize("widths", [(10,), (10, 12), (10, 2, 16)])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_push_multi_places_rows_like_separate_pushes(world, widths):
    from rl_ctr_prediction_b200 import _lib, sharded
    lib = _lib.load()
    N, B = 5003, 200
    n = B * F
    rng = np.random.default_rng(40 + world)
    ids_np = rng.integers(0, N, size=(world, n))
    ids_np[0, 0] = N + 3                                   # out of range: pushed nowhere
    ids = torch.as_tensor(ids_np).to(DEV)
    cap = sharded.route_capacity(n, world)
    _, _, wss = _route(lib, ids, world, N, cap)
    pitch = sum(widths)
    srcs = [[torch.randn(n, w, device=DEV) for w in widths] for _ in range(world)]
    multi = [torch.full((world * cap, pitch), -7.0, device=DEV) for _ in range(world)]
    single = [[torch.full((world * cap, w), -7.0, device=DEV) for _ in range(world)] for w in widths]
    mp = (C.c_void_p * 8)(*[b.data_ptr() for b in multi])
    for r in range(world):
        sp = (C.c_void_p * len(widths))(*[s.data_ptr() for s in srcs[r]])
        wd = (C.c_int32 * len(widths))(*widths)
        _lib.check(lib.rlctr_push_rows_routed_multi(_ptr(wss[r]), n, world, r, cap, sp, wd, len(widths), mp, _lib.stream()),
                   "rlctr_push_rows_routed_multi")
        for k, w in enumerate(widths):
            pp = (C.c_void_p * 8)(*[b.data_ptr() for b in single[k]])
            _lib.check(lib.rlctr_push_rows_routed(_ptr(wss[r]), n, world, r, cap, _ptr(srcs[r][k]), w, pp, _lib.stream()),
                       "rlctr_push_rows_routed")
    for o in range(world):
        want = torch.cat([single[k][o] for k in range(len(widths))], dim=1)
        assert torch.equal(multi[o], want)
        if len(widths) == 1:                               # one source, pitch = width: the old call's bytes
            assert torch.equal(multi[o].view(torch.int32), single[0][o].view(torch.int32))
    written = sum(int((m[:, 0] != -7.0).sum()) for m in multi)
    assert written == world * n - 1                        # every in-range occurrence landed once


def _member_layout(kinds):
    from rl_ctr_prediction_b200 import colocated, sharded
    ms = [sharded._dense_member(k, F, D, "cpu") for k in kinds]
    cols, used = colocated._layout(ms)
    return ms, cols, used


def _members(ms, cols, extras, pitches):
    from rl_ctr_prediction_b200 import _lib
    arr = (_lib.Member * len(ms))()
    for i, (m, (lin, emb, dim)) in enumerate(zip(ms, cols)):
        s = arr[i]
        s.lin_col, s.emb_col, s.dim = lin, emb, dim
        s.flags = _lib.RLCTR_FM_TERM if m._fm_term else 0
        s.extra = extras[i]
        s.extra_pitch = pitches[i]
    return arr


@pytest.mark.parametrize("kinds", [("DeepFM", "InnerPNN"), ("AFM", "LR", "DCN")])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_group_fwd_through_peers_equals_unsharded(world, kinds):
    from rl_ctr_prediction_b200 import _lib
    from rl_ctr_prediction_b200.tables import table_struct, Geometry
    lib = _lib.load()
    ms, cols, used = _member_layout(kinds)
    rs = (used + 1 + 3) // 4 * 4
    N, B = 4001, 300
    g = torch.Generator(device=DEV).manual_seed(world)
    full = torch.randn(N, 96, device=DEV, generator=g)
    x = torch.randint(0, N, (B, F), device=DEV, generator=g)
    x[0, 0] = N + 5                                        # out of range: a zero row

    def run(t):
        logits, rows = [], []
        arr = (_lib.Member * len(ms))()
        for i, (m, (lin, emb, dim)) in enumerate(zip(ms, cols)):
            s = arr[i]
            s.lin_col, s.emb_col, s.dim = lin, emb, dim
            s.flags = _lib.RLCTR_FM_TERM if m._fm_term else 0
            z = torch.full((B,), -3.0, device=DEV)
            s.logit = z.data_ptr()
            logits.append(z)
            r = None
            if hasattr(m, "_tail"):
                r = torch.zeros(B, (F * dim + 3) // 4 * 4, device=DEV)
                s.rows_out, s.rows_pitch = r.data_ptr(), r.shape[1]
            rows.append(r)
        sums = torch.zeros(B, 32, device=DEV)
        _lib.check(lib.rlctr_group_fwd(_ptr(x), C.byref(t), arr, len(ms), _ptr(sums), 32, B, F, _lib.stream()), "rlctr_group_fwd")
        return logits, rows, sums

    geom = Geometry(N, rs, -1, 0, used, pitch=96, block=32, stamp_at=used)
    want = run(table_struct(full, geom))
    shards = [full[r::world].contiguous() for r in range(world)]
    t = _lib.Table(shards[0].data_ptr(), N, rs, -1, 0, used, 96)
    t.world = world
    for r in range(world):
        t.peers[r] = shards[r].data_ptr()
    got = run(t)
    for a, b in zip(want[0] + want[1] + [want[2]], got[0] + got[1] + [got[2]]):
        if a is not None:
            assert torch.equal(a, b)


@pytest.mark.parametrize("kinds", [("DeepFM", "InnerPNN"), ("AFM", "LR", "DCN"), ("LR", "FM", "FNN")])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_owner_updates_with_interleaved_rows_equal_single_table(world, kinds):
    """Every owner runs rlctr_group_rows_adam(world = G, slot_of) on its shard with the interleaved receive rows of ONE multi-source
    push (extra_pitch = the row's pitch); the union of the shards and moments equals one single-table update on the concatenated
    batch, bit for bit."""
    from rl_ctr_prediction_b200 import _lib, sharded
    from rl_ctr_prediction_b200.tables import Geometry, TableAdamState, table_struct
    lib = _lib.load()
    ms, cols, used = _member_layout(kinds)
    rs = (used + 1 + 3) // 4 * 4
    N, B = 3001, 256
    n = B * F
    gen = torch.Generator(device=DEV).manual_seed(7 * world)
    per = N // F
    xs = (torch.rand(world, B, F, device=DEV, generator=gen) ** 4 * per).long() + torch.arange(F, device=DEV) * per
    ids = xs.reshape(world, n).contiguous()
    sums_all = torch.randn(world * B, 32, device=DEV, generator=gen)           # S | dL/dlogit of member m in column 28 + m
    tails = [i for i, m in enumerate(ms) if hasattr(m, "_tail")]
    grads = {i: torch.randn(world, n, cols[i][2], device=DEV, generator=gen) for i in tails}   # per-occurrence tail gradients
    init = torch.randn(N, 96, device=DEV, generator=gen)
    hyper = (1e-3, (0.9, 0.999), 1e-8, 1e-5, "lazy")

    def update(data, geom, sorted_ids, sorted_slots, n_sorted, extras, pitches, w, slot_of):
        st = TableAdamState(data, geom, *hyper)
        st.sched.ensure(4)
        arr = _members(ms, cols, extras, pitches)
        wsb = lib.rlctr_rows_ws_bytes(n_sorted)
        ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
        _lib.check(lib.rlctr_group_rows_adam(_ptr(sorted_ids), _ptr(sorted_slots), n_sorted, C.byref(table_struct(data, geom)),
                                             C.byref(st.struct()), arr, len(ms), _ptr(sums_all), 32, F, w, _ptr(slot_of), _ptr(ws),
                                             wsb, _lib.stream()), "rlctr_group_rows_adam")
        return data

    # the single table on the concatenated batch (global slot = rank * n + slot)
    geom = Geometry(N, rs, -1, 0, used, pitch=96, block=32, stamp_at=used)
    full = init.clone()
    wsb = lib.rlctr_sort_ws_bytes(world * n, N)
    ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
    sid = torch.empty(world * n, dtype=torch.int32, device=DEV)
    sslot = torch.empty(world * n, dtype=torch.int32, device=DEV)
    _lib.check(lib.rlctr_sort_ids(_ptr(ids.reshape(-1)), world * n, N, _ptr(sid), _ptr(sslot), _ptr(ws), wsb, _lib.stream()),
               "rlctr_sort_ids")
    flat = {i: grads[i].reshape(world * n, -1).contiguous() for i in tails}
    update(full, geom, sid, sslot, world * n, [_ptr(flat.get(i)) for i in range(len(ms))], [0] * len(ms), 1, None)

    # G owners: routed ids, ONE push of every tail member's rows per source, the update on each shard
    cap = sharded.route_capacity(n, world)
    keys, vals, wss = _route(lib, ids, world, N, cap)
    offs, pitch = {}, 0
    for i in tails:
        offs[i] = pitch
        pitch += cols[i][2]
    recv = [torch.zeros(world * cap * pitch, device=DEV) for _ in range(world)]
    rp = (C.c_void_p * 8)(*[b.data_ptr() for b in recv])
    for r in range(world):
        srcs = [grads[i][r].contiguous() for i in tails]
        sp = (C.c_void_p * len(srcs))(*[s.data_ptr() for s in srcs])
        wd = (C.c_int32 * len(srcs))(*[cols[i][2] for i in tails])
        _lib.check(lib.rlctr_push_rows_routed_multi(_ptr(wss[r]), n, world, r, cap, sp, wd, len(srcs), rp, _lib.stream()),
                   "rlctr_push_rows_routed_multi")
    for o in range(world):
        n_local = sharded.shard_rows(N, world, o)
        sgeom = Geometry(n_local, rs, -1, 0, used, pitch=96, block=32, stamp_at=used)
        shard = init[o::world].contiguous()
        srows = torch.empty(world * cap, dtype=torch.int32, device=DEV)
        spos = torch.empty(world * cap, dtype=torch.int32, device=DEV)
        wsb2 = lib.rlctr_sort_ws_bytes(world * cap, n_local)
        ws2 = torch.empty(wsb2, dtype=torch.uint8, device=DEV)
        _lib.check(lib.rlctr_sort_routed_pos(_ptr(keys[o]), world * cap, n_local, _ptr(srows), _ptr(spos), _ptr(ws2), wsb2,
                                             _lib.stream()), "rlctr_sort_routed_pos")
        extras = [recv[o].data_ptr() + 4 * offs[i] if i in offs else None for i in range(len(ms))]
        pitches = [pitch if i in offs else 0 for i in range(len(ms))]
        update(shard, sgeom, srows, spos, world * cap, extras, pitches, world, vals[o])
        assert torch.equal(shard, full[o::world]), o


# ---- 5. graph capture ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("names", [("LR", "FM", "FNN"), ("AFM", "LR", "DCN"), ("DeepFM", "InnerPNN")])
def test_graphed_tail_group_step_equals_eager(one_rank, names):
    from rl_ctr_prediction_b200 import colocated, graphs, optim, sharded
    N, B, steps = 4000, 256, 6
    ga = sharded.ShardedGroup.from_group(colocated.colocate(_models(names, N, seed=9, dropout=True)))
    gb = sharded.ShardedGroup.from_group(colocated.colocate(_models(names, N, seed=9, dropout=True)))
    oa = optim.Adam(ga.parameters(), lr=1e-3, weight_decay=1e-5)
    ob = optim.Adam(gb.parameters(), lr=1e-3, weight_decay=1e-5)
    step = graphs.GraphedTrainStep([(ga, oa)])
    batches = _batches(N, B, steps, seed=4)
    la = [step(x, y)[0].clone() for x, y in batches]
    lb = [gb.train_step(x, y, ob).clone() for x, y in batches]
    assert step.graph is not None
    for u, v in zip(la, lb):
        assert torch.equal(u, v)
    assert torch.equal(ga.gather_table(), gb.gather_table())
    for (ka, pa), (kb, pb) in zip(ga.named_parameters(), gb.named_parameters()):
        assert ka == kb and torch.equal(pa, pb), ka
    for a, b in zip(ga.members, gb.members):
        assert _rng_counters(a) == _rng_counters(b)


# ---- 6. errors ------------------------------------------------------------------------------------------------------------------------
def test_sharded_refusals(one_rank):
    from rl_ctr_prediction_b200 import _lib, colocated, sharded
    with pytest.raises(_lib.RlctrError):
        sharded.ShardedGroup(("LR", "FFM"), 1000, F, D)
    with pytest.raises(_lib.RlctrError):
        sharded.ShardedGroup(("AFM", "DCN", "InnerPNN"), 1000, F, D)
    with pytest.raises(_lib.RlctrError):
        sharded.ShardedCTR("NotAModel", 1000, F, D)
    cg = colocated.colocate(_models(("AFM", "LR", "DCN"), 1000, seed=1, dropout=False))
    sg = sharded.ShardedGroup.from_group(cg)
    assert [type(m).__name__ for m in sg.members] == ["AFM", "LR", "DCN"]
    assert sg.biases[2] is None and isinstance(sg.mlps[0], torch.nn.Identity)


# ---- 7. ShardedCTR.from_model carries DeepFM's dropout state -----------------------------------------------------------------------
def test_sharded_deepfm_from_model_copies_tower_dropout_state(one_rank):
    """A DeepFM whose tower is in train() and has already drawn masks (one Dropout switched to eval): the sharded copy has the
    tower's dropout counter and train / eval flags, so its first step draws the same masks and takes the same loss."""
    from rl_ctr_prediction_b200 import graphs, optim, pretrain_main as PM, sharded
    N, B = 3001, 256
    torch.manual_seed(12)
    single = PM.get_model("DeepFM", N, F, D).to(DEV).train()
    single.mlp[5].eval()
    (x0, _), (x, y) = _batches(N, B, 2, seed=13)
    with torch.no_grad():
        single(x0)                                         # the tower draws masks: its counter moves off zero
    assert int(single.mlp._rlctr_rng[1]) > 0
    m = sharded.ShardedCTR.from_model(single)
    assert torch.equal(m.mlp._rlctr_rng, single.mlp._rlctr_rng)
    assert [u.training for u in m.mlp.modules()] == [v.training for v in single.mlp.modules()]
    assert not m.mlp[5].training and m.mlp[2].training
    opt_s = optim.Adam(single.parameters(), lr=1e-3, weight_decay=1e-5)
    opt_m = optim.Adam(m.parameters(), lr=1e-3, weight_decay=1e-5)
    ls = graphs.fused_logit_step(single, opt_s, x, y)
    lm = m.train_step(x, y, opt_m)
    assert torch.equal(ls, lm)
    assert torch.equal(m.mlp._rlctr_rng, single.mlp._rlctr_rng)
