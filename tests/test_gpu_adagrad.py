"""optim.Adagrad against stock torch.optim.Adagrad driving the CPU port of the reference models (oracle/torch_port.py) at the
DESIGN.md section 4 bar (every row of every table at 2e-5, per-step losses at 1e-5), and its own paths against each other bit for
bit: lazy against dense, co-located and row-sharded records against the stand-alone model, graph replays against eager steps,
owner updates of emulated ranks against one table."""
import copy
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import torch_port as TP

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NAMES = ["LR", "FM", "FFM", "DeepFM", "W&D", "FNN", "IPNN", "OPNN", "DCN", "AFM"]
PORT_KIND = {"W&D": "WideAndDeep", "IPNN": "InnerPNN", "OPNN": "OuterPNN"}
TOWER = {"W&D", "DeepFM", "FNN", "IPNN", "OPNN", "DCN", "AFM"}
SETTINGS = {"wd0": dict(lr=1e-2), "wd": dict(lr=1e-2, weight_decay=1e-5),
            "decay": dict(lr=2e-2, lr_decay=0.05, initial_accumulator_value=0.1, weight_decay=1e-5, eps=1e-9)}


def close(a, b, rtol=2e-5):
    a, b = a.detach().cpu().double().numpy(), b.detach().cpu().double().numpy()
    np.testing.assert_allclose(a, b, rtol=rtol, atol=rtol * max(float(np.abs(b).max()), 1e-30))


def _pair(name, N, F, D, seed=3):
    from rl_ctr_prediction_b200 import pretrain_main as PM
    torch.manual_seed(seed)
    port = TP.make_port(PORT_KIND.get(name, name), N, F, D)
    with torch.no_grad():
        for k, p in port.named_parameters():
            if "embedding" in k or k == "linear.weight":
                p.mul_(0.1)
    port.eval()
    m = PM.get_model(name, N, F, D)
    m.load_state_dict(port.state_dict())
    if name == "AFM":
        port.dropout_p = m.dropout_p = 0.0
    return m.to(DEV).eval(), port


def assert_state(sd, ref_sd, tower, lr, steps, rtol=2e-5, frac=2e-3):
    """Every parameter at the bar, but for this: Adagrad's step g / sqrt(s) does not scale with g, so an element whose gradient
    nearly cancels -- its last bits set by the order of a sum -- may move by up to clr either way.  Such elements are allowed on
    at most `frac` of a table (one element of a small one), and for a model with a tower (whose GEMMs round differently from the
    CPU's) on at most `frac` of any parameter (four elements of a small one); all of them within the travel of `steps` steps."""
    assert set(sd) == set(ref_sd)
    for k, v in ref_sd.items():
        a, b = sd[k].detach().cpu().double().numpy(), v.detach().cpu().double().numpy()
        bad = np.abs(a - b) > rtol * np.abs(b) + rtol * float(np.abs(b).max())
        table = "embedding" in k or k == "linear.weight"
        allowed = max(frac * b.size, 4 if tower else 1) if (table or tower) else 0
        assert bad.sum() <= allowed, (k, int(bad.sum()), float(np.abs(a - b).max()))
        assert np.abs(a - b).max() <= 2.2 * lr * steps, k


def _batches(N, F, steps, B=64, seed=0, zipf=False, out_of_range=False):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(steps):
        x = (rng.random((B, F)) ** 6 * N).astype(np.int64).clip(0, N - 1) if zipf else rng.integers(0, N, size=(B, F))
        x[:, 1] = x[:, 0]                                             # repeated ids inside a sample
        if out_of_range:
            x[0, 0], x[-1, 2] = N + 7, -1
        out.append((torch.as_tensor(x), torch.as_tensor((rng.random(B) < 0.3).astype(np.int64)).unsqueeze(1)))
    return out


def _step(m, opt, x, y):
    p = m(x.to(DEV))
    tl = torch.nn.BCELoss()(p, y.to(DEV).float())
    m.zero_grad()
    tl.backward()
    opt.step()
    return tl.item()


def _against_oracle(name, F, D, setting, steps=4, N=300, edit_at=2, zipf=False, B=64):
    from rl_ctr_prediction_b200 import optim
    m, port = _pair(name, N, F, D)
    kw = SETTINGS[setting]
    opt = optim.Adagrad(m.parameters(), **kw)
    popt = torch.optim.Adagrad(port.parameters(), **kw)
    lossf = torch.nn.BCELoss()
    for s, (x, y) in enumerate(_batches(N, F, steps, B=B, zipf=zipf)):
        if s == edit_at:
            for o in (opt, popt):
                o.param_groups[0]["lr"] *= 0.6
        ref = TP.ctr_train_step(port, popt, lossf, x, y)
        ours = _step(m, opt, x, y)
        assert abs(ours - ref) <= 1e-5 * max(1.0, abs(ref)), (s, ours, ref)
    # every row of every table, untouched ones included
    assert_state(m.state_dict(), port.state_dict(), name in TOWER, kw["lr"], steps)
    return m


@pytest.mark.parametrize("setting", list(SETTINGS))
@pytest.mark.parametrize("name", NAMES)
def test_models_match_torch_adagrad(name, setting):
    _against_oracle(name, 15, 10, setting)


@pytest.mark.parametrize("name, F, D", [("FM", 15, 32), ("FFM", 39, 13), ("DeepFM", 15, 32)])
def test_edge_shapes_match_torch_adagrad(name, F, D):
    """36-float FM rows (the wide kernel) and FFM rows of 508 floats, with weight decay (catch-up and flush on those rows)."""
    _against_oracle(name, F, D, "wd", steps=3)


def test_zipf_heavy_hitters_match_torch_and_repeat_bit_for_bit():
    """Runs over LONG_RUN occurrences of one id go to the fixed-shape tree: torch's numbers, and the same bits every run."""
    outs = []
    for _ in range(2):
        m = _against_oracle("FM", 15, 10, "wd", steps=3, B=512, zipf=True, N=3000)
        outs.append(m.table.data.clone())
    assert torch.equal(outs[0], outs[1])


def _train(m, batches, **kw):
    from rl_ctr_prediction_b200 import _lib, optim
    opt = optim.Adagrad(m.parameters(), **kw)
    timer = _lib.KernelTimer()
    _lib.set_timer(timer)
    try:
        losses = [_step(m, opt, x, y) for x, y in batches]
        m.flush()
        torch.cuda.synchronize()
    finally:
        _lib.set_timer(None)
    return losses, set(timer.records)


@pytest.mark.parametrize("name", ["LR", "FM", "FFM", "DeepFM", "AFM"])
def test_lazy_equals_dense_bit_for_bit(name):
    """weight_decay > 0: lazy catch-up + flush == a flush after every step.  weight_decay == 0: lazy keeps no stamps and launches
    no catch-up or flush at all, and still equals the dense replay of every row every step."""
    N, F, D = 400, 15, 10
    batches = _batches(N, F, 5, seed=4, out_of_range=True)
    for wd in (1e-5, 0.0):
        a, _ = _pair(name, N, F, D)
        b, _ = _pair(name, N, F, D)
        la, keys_a = _train(a, batches, lr=2e-2, weight_decay=wd)
        lb, keys_b = _train(b, batches, lr=2e-2, weight_decay=wd, mode="dense")
        assert la == lb
        if wd:                                            # (with wd == 0 only the dense run keeps stamps in a padding column)
            assert torch.equal(a.table.data[:, :2 * a._geom.block_floats], b.table.data[:, :2 * b._geom.block_floats])
        for (k, u), (_, v) in zip(a.state_dict().items(), b.state_dict().items()):
            assert torch.equal(u, v), k
        replays = {k for k in keys_a if k.startswith(("rlctr_adagrad_catchup", "rlctr_adagrad_flush"))}
        assert bool(replays) == (wd > 0), keys_a
        assert any(k.startswith("rlctr_adagrad_flush") for k in keys_b)
        assert not any("adam" in k for k in keys_a | keys_b)


def test_optimizer_switch_adam_adagrad_adam():
    """A fresh optimizer settles what the previous one owes, then owns fresh state: Adam -> Adagrad -> Adam on one model equals
    the same sequence on the CPU port."""
    from rl_ctr_prediction_b200 import optim
    N, F, D = 300, 15, 10
    m, port = _pair("DeepFM", N, F, D)
    lossf = torch.nn.BCELoss()
    bs = _batches(N, F, 6, seed=9)
    for k, (ours_cls, ref_cls, kw) in enumerate([(optim.Adam, torch.optim.Adam, dict(lr=1e-3, weight_decay=1e-5)),
                                                 (optim.Adagrad, torch.optim.Adagrad, dict(lr=1e-2, weight_decay=1e-5)),
                                                 (optim.Adam, torch.optim.Adam, dict(lr=1e-3))]):
        opt, popt = ours_cls(m.parameters(), **kw), ref_cls(port.parameters(), **kw)
        for x, y in bs[2 * k:2 * k + 2]:
            ref = TP.ctr_train_step(port, popt, lossf, x, y)
            assert abs(_step(m, opt, x, y) - ref) <= 1e-5 * max(1.0, abs(ref))
    assert_state(m.state_dict(), port.state_dict(), True, 1e-2, 6)


def test_dense_kernel_matches_torch_adagrad():
    """rlctr_dense_adagrad_multi on replicated tensors against torch.optim.Adagrad, with a parameter that gets no gradient on some
    steps (skipped; its own step counter, so its lr_decay schedule starts late)."""
    from rl_ctr_prediction_b200 import optim
    torch.manual_seed(0)
    a0, b0 = torch.randn(40, 7), torch.randn(33)
    ours = [torch.nn.Parameter(a0.clone().to(DEV)), torch.nn.Parameter(b0.clone().to(DEV))]
    ref = [torch.nn.Parameter(a0.clone()), torch.nn.Parameter(b0.clone())]
    kw = dict(lr=0.05, lr_decay=0.1, weight_decay=1e-3, initial_accumulator_value=0.05)
    opt, ropt = optim.Adagrad(ours, **kw), torch.optim.Adagrad(ref, **kw)
    for s in range(6):
        ga, gb = torch.randn(40, 7), torch.randn(33)
        for ps in (ours, ref):
            ps[0].grad = ga.clone().to(ps[0].device)
            ps[1].grad = gb.clone().to(ps[1].device) if s >= 2 and s != 4 else None
        if s == 3:
            for o in (opt, ropt):
                o.param_groups[0]["lr"] = 0.02
        opt.step()
        ropt.step()
        close(ours[0], ref[0], 1e-6)
        close(ours[1], ref[1], 1e-6)
    assert opt._dense_count == [6, 3] and opt._dense_steps.tolist() == [6, 3]


def _models(N, F, D, names, seed=3):
    from rl_ctr_prediction_b200 import pretrain_main as PM
    torch.manual_seed(seed)
    ms = [PM.get_model(n, N, F, D).to(DEV).train() for n in names]
    for m in ms:
        if getattr(m, "mlp", None) is not None:
            m.mlp.eval()
    return ms


def _group_batches(N, F, B, steps, seed=11, zipf=False):
    g = torch.Generator().manual_seed(seed)
    per = N // F
    out = []
    for _ in range(steps):
        x = (torch.rand(B, F, generator=g) ** 6 * per).long().clamp_(0, per - 1) if zipf else torch.randint(0, per, (B, F), generator=g)
        x = x + torch.arange(F) * per
        x[0, 0] = N + 3                                   # out of range: zero row, no update
        out.append((x.to(DEV), (torch.rand(B, generator=g) < 0.3).long().to(DEV)))
    return out


@pytest.mark.parametrize("wd", [0.0, 1e-5])
@pytest.mark.parametrize("names, D, max_lines", [(("LR", "FM", "DeepFM"), 10, 1), (("LR", "FM", "DeepFM"), 32, 4)])
def test_group_equals_standalone_models(names, D, max_lines, wd):
    from rl_ctr_prediction_b200 import colocated, graphs, optim
    N, F, B, steps = 3000, 15, 512, 5
    sep = _models(N, F, D, names)
    grp = [copy.deepcopy(m) for m in sep]
    batches = _group_batches(N, F, B, steps, zipf=True)
    kw = dict(lr=1e-2, weight_decay=wd)
    opts = [optim.Adagrad(m.parameters(), **kw) for m in sep]
    lossf = torch.nn.BCELoss()
    l_sep = np.array([[float(graphs.eager_step(m, o, lossf, x, y)) for m, o in zip(sep, opts)] for x, y in batches])
    group = colocated.colocate(grp, max_lines=max_lines)
    assert (group._geom.row_pitch == 96) == (max_lines == 1)
    opt = optim.Adagrad(group.parameters(), **kw)
    l_grp = np.array([group.train_step(x, y, opt).cpu().numpy().copy() for x, y in batches])
    assert np.array_equal(l_sep[:, 1:], l_grp[:, 1:])
    np.testing.assert_allclose(l_grp[:, 0], l_sep[:, 0], rtol=2e-6)
    for i, name in enumerate(names):
        a, b = sep[i].state_dict(), grp[i].state_dict()
        for k in a:
            if name == "LR":
                torch.testing.assert_close(b[k], a[k], rtol=0, atol=2e-6)
            else:
                assert torch.equal(a[k], b[k]), (name, k)


@pytest.fixture(scope="module")
def one_rank():
    import torch.distributed as dist
    if not dist.is_initialized():
        import socket
        s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
        dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=0, world_size=1, device_id=torch.device(DEV))
    yield None
    if dist.is_initialized():
        dist.destroy_process_group()


@pytest.mark.parametrize("wd", [0.0, 1e-5])
@pytest.mark.parametrize("name", ["LR", "FM", "FFM", "DeepFM"])
def test_sharded_world1_equals_single_gpu(one_rank, name, wd):
    from rl_ctr_prediction_b200 import optim, pretrain_main, sharded
    N, F, D = 500, 15, 10
    single, _ = _pair(name, N, F, D)
    twin = copy.deepcopy(single)
    m = sharded.ShardedCTR.from_model(twin)
    m.eval()
    kw = dict(lr=1e-2, weight_decay=wd)
    o1, o2 = optim.Adagrad(single.parameters(), **kw), optim.Adagrad(m.parameters(), **kw)
    for x, y in _batches(N, F, 4, seed=2):
        x, y = x.to(DEV), y.to(DEV)
        l1 = float(pretrain_main.fused_train_step(single, o1, x, y))
        l2 = float(m.train_step(x, y, o2))
        assert l1 == l2
    single.flush()
    assert torch.equal(m.gather_table(), single.table.data)
    assert torch.equal(m.bias.data, single.bias.data)


@pytest.mark.parametrize("wd", [0.0, 1e-5])
def test_sharded_group_world1_equals_colocated(wd):
    from rl_ctr_prediction_b200 import colocated, optim, sharded
    N, F, D, B = 3001, 15, 10, 384
    cg = colocated.colocate(_models(N, F, D, ("LR", "FM", "DeepFM"), seed=21))
    sg = sharded.ShardedGroup.from_group(cg)
    for mlp in sg.mlps:
        mlp.eval()
    oa, ob = optim.Adagrad(cg.parameters(), lr=1e-2, weight_decay=wd), optim.Adagrad(sg.parameters(), lr=1e-2, weight_decay=wd)
    for x, y in _group_batches(N, F, B, 4, seed=6, zipf=True):
        assert torch.equal(cg.train_step(x, y, oa), sg.train_step(x, y, ob))
    cg.flush()
    assert torch.equal(sg.gather_table()[:, :64], cg.table.data[:, :64])


@pytest.mark.parametrize("wd", [0.0, 1e-5])
def test_graphed_replays_equal_eager_steps_and_see_lr_edits(wd):
    from rl_ctr_prediction_b200 import graphs, optim
    N, F, D, B, steps = 3000, 15, 10, 256, 7
    a = _models(N, F, D, ("LR", "FM", "DeepFM"), seed=5)
    b = _models(N, F, D, ("LR", "FM", "DeepFM"), seed=5)
    batches = _group_batches(N, F, B, steps, seed=4)
    oa = [optim.Adagrad(m.parameters(), lr=1e-2, weight_decay=wd) for m in a]
    ob = [optim.Adagrad(m.parameters(), lr=1e-2, weight_decay=wd) for m in b]
    step = graphs.GraphedTrainStep(list(zip(a, oa)))
    lossf = torch.nn.BCELoss()
    la, lb = [], []
    for s, (x, y) in enumerate(batches):
        if s == 5:                                        # an lr edit between replays takes effect in the captured graph
            for o in oa + ob:
                o.param_groups[0]["lr"] = 3e-3
        la.append([float(v) for v in step(x, y)])
        lb.append([float(graphs.eager_step(m, o, lossf, x, y)) for m, o in zip(b, ob)])
    assert step.graph is not None
    assert la == lb
    for u, v in zip(a, b):
        for (k, p), (_, q) in zip(u.state_dict().items(), v.state_dict().items()):
            assert torch.equal(p, q), k


def _L():
    from rl_ctr_prediction_b200 import _lib
    return _lib


@pytest.mark.parametrize("wd", [0.0, 1e-5])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_emulated_ranks_equal_one_table(world, wd):
    """G ranks emulated on one GPU: each owner runs rlctr_rows_adagrad (FM rows) and rlctr_group_rows_adagrad (a one-line
    co-located record) on its shard with the peer gradient buffers; the union of the shards equals the unsharded call bit for bit."""
    from rl_ctr_prediction_b200 import sharded
    from rl_ctr_prediction_b200.tables import AdagradSchedule
    L = _L()
    lib = L.load()
    st = L.stream()
    N, B, F, D = 3001, 200, 15, 10
    rng = np.random.default_rng(7 + world)
    sched = AdagradSchedule(1e-2, 0.01, DEV)
    ids = rng.integers(0, N, size=(world, B, F))
    ids[:, :, 1] = ids[:, :, 0]
    dl = [rng.standard_normal(B).astype(np.float32) * 0.1 for _ in range(world)]
    ex = [rng.standard_normal((B, F * D)).astype(np.float32) * 0.1 for _ in range(world)]
    x_all = torch.as_tensor(ids.reshape(-1, F)).to(DEV)
    n_all = x_all.numel()

    def sorted_all():
        sid, ssl = torch.empty(n_all, dtype=torch.int32, device=DEV), torch.empty(n_all, dtype=torch.int32, device=DEV)
        wsb = lib.rlctr_sort_ws_bytes(n_all, N)
        ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
        L.check(lib.rlctr_sort_ids(L.ptr(x_all), n_all, N, L.ptr(sid), L.ptr(ssl), L.ptr(ws), wsb, st), "sort")
        return sid, ssl

    def sorted_owned(rank):
        all32 = x_all.reshape(-1).to(torch.int32)
        srows, sslots = torch.empty(n_all, dtype=torch.int32, device=DEV), torch.empty(n_all, dtype=torch.int32, device=DEV)
        wsb = lib.rlctr_sort_ws_bytes(n_all, N)
        ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
        L.check(lib.rlctr_sort_ids_sharded(L.ptr(all32), n_all, world, rank, N, L.ptr(srows), L.ptr(sslots), L.ptr(ws), wsb, st), "s")
        return srows, sslots

    rwb = lib.rlctr_rows_ws_bytes(n_all)
    rws = torch.empty(rwb, dtype=torch.uint8, device=DEV)
    for kind in ("rows", "group"):
        rs, pitch = (16, 48) if kind == "rows" else (24, 96)
        blk = rs if kind == "rows" else 32
        full = np.zeros((N, pitch), np.float32)
        full[:, :11] = rng.standard_normal((N, 11)).astype(np.float32) * 0.1
        full[:, blk:blk + rs] = 0.05                                      # initial_accumulator_value
        stamp_col = 11 if wd else -1
        full[:, 11] = 0
        sums = [rng.standard_normal((B, rs)).astype(np.float32) for _ in range(world)]

        def run(tab, n_rows, sid, ssl, gworld, bufs):
            step = torch.full((1,), 3, dtype=torch.int32, device=DEV)    # three completed steps: the wd replay has work
            a = L.Adagrad(tab.data_ptr() + 4 * blk, None, L.ptr(sched.tensor), L.ptr(step), sched.length, stamp_col, 1e-10, wd)
            t = L.Table(L.ptr(tab), n_rows, rs, 0 if kind == "rows" else -1, 1 if kind == "rows" else 0, D if kind == "rows" else 11,
                        pitch)
            if kind == "rows":
                g = L.RowGrad(None, None, None, None, F, 0)
                g.world, g.n_per_rank = gworld, B * F
                if gworld > 1:
                    for r in range(gworld):
                        g.peer_dlogit[r], g.peer_sums[r], g.peer_extra[r] = [u.data_ptr() for u in bufs[r]]
                else:
                    g.dlogit, g.sums, g.extra = [u.data_ptr() for u in bufs[0]]
                L.check(lib.rlctr_rows_adagrad(L.ptr(sid), L.ptr(ssl), n_all, C.byref(g), C.byref(t), C.byref(a), L.ptr(rws), rwb, st),
                        "rows")
            else:
                mem = (L.Member * 2)()
                mem[0].lin_col, mem[0].emb_col, mem[0].dim, mem[0].dlogit = 0, 0, 0, bufs[0].data_ptr()
                mem[1].lin_col, mem[1].emb_col, mem[1].dim, mem[1].flags = 1, 2, 9, 1
                mem[1].dlogit = bufs[0].data_ptr()
                L.check(lib.rlctr_group_rows_adagrad(L.ptr(sid), L.ptr(ssl), n_all, C.byref(t), C.byref(a), mem, 2, L.ptr(bufs[1]), 0,
                                                     F, gworld, None, L.ptr(rws), rwb, st), "group")

        tab = torch.as_tensor(full).to(DEV)
        sid, ssl = sorted_all()
        if kind == "rows":
            run(tab, N, sid, ssl, 1, [[torch.as_tensor(np.concatenate(v)).to(DEV) for v in (dl, sums, ex)]])
            bufs = [[torch.as_tensor(v[r]).to(DEV) for v in (dl, sums, ex)] for r in range(world)]
        else:
            gbufs = [torch.as_tensor(np.concatenate(dl)).to(DEV), torch.as_tensor(np.concatenate(sums)).to(DEV)]
            run(tab, N, sid, ssl, 1, gbufs)
        for rank in range(world):
            shard = torch.as_tensor(full[rank::world].copy()).to(DEV)
            srows, sslots = sorted_owned(rank)
            run(shard, sharded.shard_rows(N, world, rank), srows, sslots, world, bufs if kind == "rows" else gbufs)
            assert torch.equal(shard, tab[rank::world]), (kind, rank)
