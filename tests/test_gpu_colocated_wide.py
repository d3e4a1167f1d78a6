"""Co-located records wider than one 128-byte line (colocate(..., max_lines=2..4), sharded.ShardedGroup(..., max_lines=...)).

A wide joint row holds up to 128 floats: three or four vector members, latent sizes past 14, members whose stand-alone rows are
20 to 36 floats.  Every vector member must give the numbers of its stand-alone model bit for bit -- losses, every row of its table
after the flush, every dense parameter, the dropout counters -- in lazy and dense Adam, with uniform ids (short runs) and Zipf ids
(runs past 32 occurrences: the stand-alone long-run trees).  LR agrees to rounding, as in the one-line groups.
"""
import copy
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
NAMES = {"LR": "LR", "FM": "FM", "DeepFM": "DeepFM", "WideAndDeep": "W&D", "FNN": "FNN", "InnerPNN": "IPNN", "OuterPNN": "OPNN",
         "DCN": "DCN", "AFM": "AFM"}
GROUPS = [(("LR", "FM", "DeepFM"), d) for d in (12, 15, 16, 20, 31, 32)] + [
    (("FM", "FNN", "DeepFM"), 10), (("LR", "OuterPNN", "FNN", "WideAndDeep"), 10), (("AFM", "DCN", "InnerPNN"), 10),
    (("FM", "FNN"), 16), (("DeepFM", "DCN"), 32)]


def _towers(m):
    from rl_ctr_prediction_b200 import mlp
    return [t for t in m.modules() if isinstance(t, mlp.Tower)]


def _set_dropout(m, seed):
    for k, t in enumerate(_towers(m)):
        t.train(True)
        t._rlctr_rng = torch.tensor([seed + 17 * k, 0], dtype=torch.int64, device=DEV)
    if type(m).__name__ == "AFM":
        m.dropout_p = 0.2
        m._rlctr_rng = torch.tensor([seed + 101, 0], dtype=torch.int64, device=DEV)


def _rng_counters(m):
    out = [int(t._rlctr_rng[1]) for t in _towers(m)]
    if type(m).__name__ == "AFM":
        out.append(int(m._rlctr_rng[1]))
    return out


def _models(names, N, F, D, seed=3):
    from rl_ctr_prediction_b200 import pretrain_main as PM
    torch.manual_seed(seed)
    ms = [PM.get_model(NAMES[n], N, F, D).to(DEV).train() for n in names]
    for i, m in enumerate(ms):
        _set_dropout(m, 1000 * seed + 10 * i)
    return ms


def _batches(N, F, B, steps, seed=11, zipf=False):
    g = torch.Generator().manual_seed(seed)
    per = N // F
    out = []
    for _ in range(steps):
        if zipf:
            x = (torch.rand(B, F, generator=g) ** 6 * per).long().clamp_(0, per - 1)     # heavy hitters: long runs of one id
        else:
            x = torch.randint(0, per, (B, F), generator=g)
        x = x + torch.arange(F) * per
        y = (torch.rand(B, generator=g) < 0.3).long()
        out.append((x.to(DEV), y.to(DEV)))
    return out


def _train_separate(models, batches, mode="lazy"):
    from rl_ctr_prediction_b200 import graphs, optim
    opts = [optim.Adam(m.parameters(), lr=1e-3, weight_decay=1e-5, mode=mode) for m in models]
    loss_fn = torch.nn.BCELoss()
    return np.array([[float(graphs.eager_step(m, o, loss_fn, x, y)) for m, o in zip(models, opts)] for x, y in batches])


def _train_group(models, batches, mode="lazy", max_lines=4):
    from rl_ctr_prediction_b200 import colocated, optim
    group = colocated.colocate(models, max_lines=max_lines)
    opt = optim.Adam(group.parameters(), lr=1e-3, weight_decay=1e-5, mode=mode)
    losses = [group.train_step(x, y, opt).cpu().numpy().copy() for x, y in batches]
    return group, np.array(losses)


def _assert_same(names, sep, grp, l_sep, l_grp):
    for i, n in enumerate(names):
        if n == "LR":
            np.testing.assert_allclose(l_grp[:, i], l_sep[:, i], rtol=2e-6)
        else:
            assert np.array_equal(l_sep[:, i], l_grp[:, i]), n
        a, b = sep[i].state_dict(), grp[i].state_dict()
        assert set(a) == set(b)
        for k in a:
            if n == "LR":
                torch.testing.assert_close(b[k], a[k], rtol=0, atol=2e-6)
            else:
                assert torch.equal(a[k], b[k]), (n, k)
        assert _rng_counters(sep[i]) == _rng_counters(grp[i]), n


@pytest.mark.parametrize("mode", ["lazy", "dense"])
@pytest.mark.parametrize("zipf", [False, True])
@pytest.mark.parametrize("names,D", GROUPS)
def test_wide_group_equals_standalone(names, D, zipf, mode):
    F, N, B, steps = 15, 3000, 512, 4
    sep = _models(names, N, F, D)
    grp = [copy.deepcopy(m) for m in sep]
    batches = _batches(N, F, B, steps, zipf=zipf)
    l_sep = _train_separate(sep, batches, mode)
    _, l_grp = _train_group(grp, batches, mode)
    _assert_same(names, sep, grp, l_sep, l_grp)


def test_wide_record_geometry():
    """Packed [p | exp_avg | exp_avg_sq] blocks, the pitch in whole lines, the stamp in the last active chunk."""
    N = 1000
    group = _train_group(_models(("LR", "FM", "DeepFM"), N, 15, 32), [])[0]
    g = group._geom
    assert (g.row_stride, g.block_floats, g.row_pitch, g.stamp_col) == (72, 72, 224, 69)
    assert group.table.shape == (N, 224)


def test_wide_graphed_step_equals_eager():
    from rl_ctr_prediction_b200 import colocated, graphs, optim
    names, F, D, N, B, steps = ("LR", "FM", "FNN", "DeepFM"), 15, 16, 4000, 256, 6
    a = _models(names, N, F, D, seed=9)
    b = [copy.deepcopy(m) for m in a]
    batches = _batches(N, F, B, steps, seed=4, zipf=True)
    ga, gb = colocated.colocate(a, max_lines=4), colocated.colocate(b, max_lines=4)
    oa = optim.Adam(ga.parameters(), lr=1e-3, weight_decay=1e-5)
    ob = optim.Adam(gb.parameters(), lr=1e-3, weight_decay=1e-5)
    step = graphs.GraphedTrainStep([(ga, oa)])
    la = [step(x, y)[0].clone() for x, y in batches]
    lb = [gb.train_step(x, y, ob).clone() for x, y in batches]
    assert step.graph is not None
    for u, v in zip(la, lb):
        assert torch.equal(u, v)
    ga.flush()
    gb.flush()
    assert torch.equal(ga.table.data, gb.table.data)
    for pa, pb in zip(ga.parameters(), gb.parameters()):
        assert torch.equal(pa, pb)


def test_wide_inference_member_views_and_state_dict():
    """group(x), each member's own forward on its stand-alone view of the record, and reference-keyed state_dict round trips."""
    from rl_ctr_prediction_b200 import pretrain_main as PM
    names, F, D, N = ("LR", "FM", "DeepFM", "FNN"), 15, 20, 3000
    sep = _models(names, N, F, D)
    grp = [copy.deepcopy(m) for m in sep]
    batches = _batches(N, F, 384, 3, zipf=True)
    _train_separate(sep, batches)
    group, _ = _train_group(grp, batches)
    for m in sep + grp:
        m.eval()
    x = _batches(N, F, 300, 1, seed=5)[0][0]
    with torch.no_grad():
        want = torch.stack([m(x).reshape(-1) for m in sep], 1)
        got = group(x)
        own = torch.stack([m(x).reshape(-1) for m in grp], 1)
    assert torch.equal(got[:, 1:], want[:, 1:]) and torch.equal(own[:, 1:], want[:, 1:])
    torch.testing.assert_close(got[:, 0], want[:, 0], rtol=2e-6, atol=0)
    for n, m in zip(names, grp):
        fresh = PM.get_model(NAMES[n], N, F, D).to(DEV)
        fresh.load_state_dict(m.state_dict())
        for k, v in m.state_dict().items():
            assert torch.equal(fresh.state_dict()[k], v), (n, k)
        m.load_state_dict(fresh.state_dict())              # and back into the joint record
        for k, v in fresh.state_dict().items():
            assert torch.equal(m.state_dict()[k], v), (n, k)


def test_wide_group_with_more_than_sixteen_fields():
    F, D, N, B, steps = 20, 16, 4000, 300, 4
    names = ("LR", "FM", "DeepFM")
    sep = _models(names, N, F, D, seed=17)
    grp = [copy.deepcopy(m) for m in sep]
    batches = _batches(N, F, B, steps, seed=23, zipf=True)
    l_sep = _train_separate(sep, batches)
    _, l_grp = _train_group(grp, batches)
    _assert_same(names, sep, grp, l_sep, l_grp)


@pytest.mark.parametrize("B", [1, 33])
def test_wide_group_ragged_batches_and_out_of_range_ids(B):
    F, D, N, steps = 15, 24, 500, 3
    names = ("LR", "FM", "DeepFM")
    sep = _models(names, N, F, D, seed=41)
    grp = [copy.deepcopy(m) for m in sep]
    g = torch.Generator().manual_seed(3)
    batches = []
    for _ in range(steps):
        x = torch.randint(0, N, (B, F), generator=g)
        x[0, 0] = N + 7                                   # out of range
        x[-1, 3] = -1
        batches.append((x.to(DEV), (torch.rand(B, generator=g) < 0.5).long().to(DEV)))
    l_sep = _train_separate(sep, batches)
    _, l_grp = _train_group(grp, batches)
    _assert_same(names, sep, grp, l_sep, l_grp)


def test_one_line_group_keeps_its_record():
    """max_lines only sets a ceiling: a group that fits one line keeps the one-line record and its bits."""
    from rl_ctr_prediction_b200 import colocated
    names, F, D, N = ("LR", "FM", "DeepFM"), 15, 10, 2000
    a, b = _models(names, N, F, D), _models(names, N, F, D)
    batches = _batches(N, F, 256, 3, zipf=True)
    ga, la = _train_group(a, batches, max_lines=1)
    gb, lb = _train_group(b, batches, max_lines=4)
    assert (gb._geom.row_stride, gb._geom.row_pitch, gb._geom.block_floats) == (24, 96, 32) == \
        (ga._geom.row_stride, ga._geom.row_pitch, ga._geom.block_floats)
    assert np.array_equal(la, lb)
    ga.flush()
    gb.flush()
    assert torch.equal(ga.table.data, gb.table.data)


# ---- row-sharded: world 1 ------------------------------------------------------------------------------------------------------
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


@pytest.mark.parametrize("mode", ["lazy", "dense"])
@pytest.mark.parametrize("names,D", [(("LR", "FM", "DeepFM"), 12), (("FM", "FNN", "DeepFM", "AFM"), 16),
                                     (("DeepFM", "DCN"), 32)])
def test_world1_wide_sharded_group_equals_colocated(one_rank, names, D, mode):
    from rl_ctr_prediction_b200 import colocated, optim, sharded
    F, N, B, steps = 15, 3001, 384, 4
    cg = colocated.colocate(_models(names, N, F, D, seed=21), max_lines=4)
    sg = sharded.ShardedGroup.from_group(cg)
    assert sg.SUMS_PITCH >= cg._geom.row_stride + 4 and sg.SUMS_PITCH % 32 == 0
    oa = optim.Adam(cg.parameters(), lr=1e-3, weight_decay=1e-5, mode=mode)
    ob = optim.Adam(sg.parameters(), lr=1e-3, weight_decay=1e-5, mode=mode)
    for x, y in _batches(N, F, B, steps, seed=6, zipf=True):
        assert torch.equal(cg.train_step(x, y, oa), sg.train_step(x, y, ob))
    cg.flush()
    assert torch.equal(sg.gather_table(), cg.table.data)
    for a, b in zip(sg.members, cg.members):
        pa = {k: p for k, p in a.named_parameters() if k != "table"}
        pb = {k: p for k, p in b.named_parameters() if k != "table"}
        assert set(pa) == set(pb)
        for k in pb:
            assert torch.equal(pa[k], pb[k]), (type(b).__name__, k)
        assert _rng_counters(a) == _rng_counters(b)
    x = _batches(N, F, B, 1, seed=8)[0][0]
    assert torch.equal(sg(x), cg(x))


def test_load_embedding_into_a_wide_member():
    """FNN.load_embedding (and the PNNs') writes the member's own columns of the joint record, not the record's first ones."""
    from rl_ctr_prediction_b200 import colocated
    names, F, D, N = ("LR", "FM", "FNN", "InnerPNN"), 15, 16, 2000
    ms = _models(names, N, F, D)
    group = colocated.colocate(ms, max_lines=4)
    before = [m.state_dict() for m in ms]
    for i in (2, 3):                                       # FNN at the record's columns 20.., InnerPNN after it
        assert ms[i]._geom.offset > 0
        ckpt = {"feature_embedding.weight": torch.randn(N, D, device=DEV)}
        ms[i].load_embedding(ckpt)
        assert torch.equal(ms[i].state_dict()["feature_embedding.weight"], ckpt["feature_embedding.weight"])
        for j in range(len(ms)):
            if j != i:
                for k, v in ms[j].state_dict().items():
                    assert torch.equal(v, before[j][k]), (names[j], k)
        before[i] = ms[i].state_dict()
    assert group._geom.row_stride > 32


def test_wide_graphed_step_with_large_tower_tiles():
    """Three tail members at D = 32: the gather's tower tiles take more than 48 KB of shared memory per block; the captured step
    equals the eager one."""
    from rl_ctr_prediction_b200 import colocated, graphs, optim
    names, F, D, N, B, steps = ("DeepFM", "FNN", "DCN"), 15, 32, 3000, 256, 4
    a = _models(names, N, F, D, seed=13)
    b = [copy.deepcopy(m) for m in a]
    batches = _batches(N, F, B, steps, seed=2, zipf=True)
    ga, gb = colocated.colocate(a, max_lines=4), colocated.colocate(b, max_lines=4)
    oa = optim.Adam(ga.parameters(), lr=1e-3, weight_decay=1e-5)
    ob = optim.Adam(gb.parameters(), lr=1e-3, weight_decay=1e-5)
    step = graphs.GraphedTrainStep([(ga, oa)])
    la = [step(x, y)[0].clone() for x, y in batches]
    lb = [gb.train_step(x, y, ob).clone() for x, y in batches]
    assert step.graph is not None
    for u, v in zip(la, lb):
        assert torch.equal(u, v)
    ga.flush()
    gb.flush()
    assert torch.equal(ga.table.data, gb.table.data)
    for pa, pb in zip(ga.parameters(), gb.parameters()):
        assert torch.equal(pa, pb)


# ---- row-sharded: G ranks emulated on one GPU -----------------------------------------------------------------------------------
EMULATED = [(("LR", "FM", "DeepFM"), 16), (("LR", "FM", "DeepFM"), 32), (("FM", "FNN"), 16), (("DeepFM", "FNN", "DCN"), 20)]


def _ptr(t):
    return t.data_ptr() if t is not None else None


def _wide_layout(kinds, F, D):
    from rl_ctr_prediction_b200 import colocated, sharded
    ms = [sharded._dense_member(k, F, D, "cpu") for k in kinds]
    cols, used = colocated._layout(ms, 4)
    return ms, cols, used, colocated._record(1, used)


def _route(lib, ids, world, N, cap):
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


@pytest.mark.parametrize("kinds,D", EMULATED)
@pytest.mark.parametrize("world", [2, 4, 8])
def test_wide_group_fwd_through_peers_equals_unsharded(world, kinds, D):
    from rl_ctr_prediction_b200 import _lib
    from rl_ctr_prediction_b200.tables import table_struct, Geometry
    lib = _lib.load()
    F = 15
    ms, cols, used, rec = _wide_layout(kinds, F, D)
    rs, pitch = rec.row_stride, rec.row_pitch
    sp = (rs + _lib.RLCTR_GROUP_MAX + 31) // 32 * 32
    N, B = 4001, 300
    g = torch.Generator(device=DEV).manual_seed(world)
    full = torch.randn(N, pitch, device=DEV, generator=g)
    per = N // F
    x = (torch.rand(B, F, device=DEV, generator=g) ** 6 * per).long() + torch.arange(F, device=DEV) * per
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
        sums = torch.zeros(B, sp, device=DEV)
        _lib.check(lib.rlctr_group_fwd(_ptr(x), C.byref(t), arr, len(ms), _ptr(sums), sp, B, F, _lib.stream()), "rlctr_group_fwd")
        return logits, rows, sums

    geom = Geometry(N, rs, -1, 0, used, pitch=pitch, block=rec.block_floats, stamp_at=used)
    want = run(table_struct(full, geom))
    shards = [full[r::world].contiguous() for r in range(world)]
    t = _lib.Table(shards[0].data_ptr(), N, rs, -1, 0, used, pitch)
    t.world = world
    for r in range(world):
        t.peers[r] = shards[r].data_ptr()
    got = run(t)
    for a, b in zip(want[0] + want[1] + [want[2]], got[0] + got[1] + [got[2]]):
        if a is not None:
            assert torch.equal(a, b)


@pytest.mark.parametrize("kinds,D", EMULATED)
@pytest.mark.parametrize("world", [2, 4, 8])
def test_wide_owner_updates_equal_single_table(world, kinds, D):
    """Every owner runs rlctr_group_rows_adam(world = G, slot_of) on its shard of wide records, with the interleaved receive rows of
    ONE multi-source push and the widened exchange rows; the union of the shards equals one single-table update on the
    concatenated batch, bit for bit.  Zipf ids: the owned long runs take group_long_wide_kernel."""
    from rl_ctr_prediction_b200 import _lib, sharded
    from rl_ctr_prediction_b200.tables import Geometry, TableAdamState, table_struct
    lib = _lib.load()
    F = 15
    ms, cols, used, rec = _wide_layout(kinds, F, D)
    rs, pitch_r, blk = rec.row_stride, rec.row_pitch, rec.block_floats
    sp = (rs + _lib.RLCTR_GROUP_MAX + 31) // 32 * 32
    N, B = 3001, 256
    n = B * F
    gen = torch.Generator(device=DEV).manual_seed(7 * world)
    per = N // F
    xs = (torch.rand(world, B, F, device=DEV, generator=gen) ** 4 * per).long() + torch.arange(F, device=DEV) * per
    ids = xs.reshape(world, n).contiguous()
    sums_all = torch.randn(world * B, sp, device=DEV, generator=gen)           # S | dL/dlogit of member m in column sp - 4 + m
    tails = [i for i, m in enumerate(ms) if hasattr(m, "_tail")]
    grads = {i: torch.randn(world, n, cols[i][2], device=DEV, generator=gen) for i in tails}
    init = torch.randn(N, pitch_r, device=DEV, generator=gen)
    hyper = (1e-3, (0.9, 0.999), 1e-8, 1e-5, "lazy")

    def members(extras, pitches):
        arr = (_lib.Member * len(ms))()
        for i, (m, (lin, emb, dim)) in enumerate(zip(ms, cols)):
            s = arr[i]
            s.lin_col, s.emb_col, s.dim = lin, emb, dim
            s.flags = _lib.RLCTR_FM_TERM if m._fm_term else 0
            s.extra = extras[i]
            s.extra_pitch = pitches[i]
        return arr

    def update(data, geom, sorted_ids, sorted_slots, n_sorted, extras, pitches, w, slot_of):
        st = TableAdamState(data, geom, *hyper)
        st.sched.ensure(4)
        wsb = lib.rlctr_rows_ws_bytes(n_sorted)
        ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
        _lib.check(lib.rlctr_group_rows_adam(_ptr(sorted_ids), _ptr(sorted_slots), n_sorted, C.byref(table_struct(data, geom)),
                                             C.byref(st.struct()), members(extras, pitches), len(ms), _ptr(sums_all), sp, F, w,
                                             _ptr(slot_of), _ptr(ws), wsb, _lib.stream()), "rlctr_group_rows_adam")

    geom = Geometry(N, rs, -1, 0, used, pitch=pitch_r, block=blk, stamp_at=used)
    full = init.clone()
    wsb = lib.rlctr_sort_ws_bytes(world * n, N)
    ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
    sid = torch.empty(world * n, dtype=torch.int32, device=DEV)
    sslot = torch.empty(world * n, dtype=torch.int32, device=DEV)
    _lib.check(lib.rlctr_sort_ids(_ptr(ids.reshape(-1)), world * n, N, _ptr(sid), _ptr(sslot), _ptr(ws), wsb, _lib.stream()),
               "rlctr_sort_ids")
    flat = {i: grads[i].reshape(world * n, -1).contiguous() for i in tails}
    update(full, geom, sid, sslot, world * n, [_ptr(flat.get(i)) for i in range(len(ms))], [0] * len(ms), 1, None)

    cap = sharded.route_capacity(n, world)
    keys, vals, wss = _route(lib, ids, world, N, cap)
    offs, pitch = {}, 0
    for i in tails:
        offs[i] = pitch
        pitch += cols[i][2]
    recv = [torch.zeros(world * cap * max(pitch, 2), device=DEV) for _ in range(world)]
    if tails:
        rp = (C.c_void_p * 8)(*[b.data_ptr() for b in recv])
        for r in range(world):
            srcs = [grads[i][r].contiguous() for i in tails]
            spp = (C.c_void_p * len(srcs))(*[s.data_ptr() for s in srcs])
            wd = (C.c_int32 * len(srcs))(*[cols[i][2] for i in tails])
            _lib.check(lib.rlctr_push_rows_routed_multi(_ptr(wss[r]), n, world, r, cap, spp, wd, len(srcs), rp, _lib.stream()),
                       "rlctr_push_rows_routed_multi")
    for o in range(world):
        n_local = sharded.shard_rows(N, world, o)
        sgeom = Geometry(n_local, rs, -1, 0, used, pitch=pitch_r, block=blk, stamp_at=used)
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
