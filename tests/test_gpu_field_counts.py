"""Every model at field counts past the reference's iPinYou encoding (F = 15): Avazu-like F = 24, Criteo's F = 39, and F = 64.

F = 24..64 reach the 16-bit pair-index backward of InnerPNN's pair dots (rlctr_pairdots_bwd; shared memory past 48 KB from
F = 64, D = 32), and F = 33..64 the one-warp FFM forward kernels (rlctr_ffm_fwd: two ids per lane, double-buffered where two
[F][row] stage buffers fit in 227 KB, single-buffered where they do not), which also take F <= 32 shapes whose stage buffers
exceed the two-warp kernel's 200 KB (F = 32 at D = 12).  Everything else (the K1 gather past 16 fields, the co-located gathers,
the row update, the tower GEMMs at K = F*D + P, the policy nets' F(F-1)/2 + F*D inputs) is exercised at those shapes against
the CPU port of the reference (oracle/torch_port.py) with the scheme and bars of tests/test_gpu_latent_dims.py."""
import copy
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import torch_port as TP

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
NAMES = ["LR", "FM", "FFM", "W&D", "DeepFM", "FNN", "IPNN", "OPNN", "DCN"]
PORT_KIND = {"W&D": "WideAndDeep", "IPNN": "InnerPNN", "OPNN": "OuterPNN"}
TOWER = {"W&D", "DeepFM", "FNN", "IPNN", "OPNN", "DCN"}


def close(a, b, rtol=1e-5, atol=None):
    """|a - b| <= rtol * max(|b|, scale of b) (tests/test_gpu_models.py's bar)."""
    a = a.detach().cpu().double().numpy() if isinstance(a, torch.Tensor) else np.asarray(a, np.float64)
    b = b.detach().cpu().double().numpy() if isinstance(b, torch.Tensor) else np.asarray(b, np.float64)
    if atol is None:
        atol = rtol * (np.abs(b).max() if b.size else 0.0)
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol)


def assert_state(sd, ref_sd, tower=False, steps=3, rtol=2e-5, table_frac=1e-4):
    """tests/test_gpu_latent_dims.py's criterion: every parameter at the parity bar; for a tower model, table elements off the
    bar on at most `table_frac` of the table and all inside Adam's travel band."""
    assert set(sd.keys()) == set(ref_sd.keys())
    for k, v in ref_sd.items():
        assert tuple(sd[k].shape) == tuple(v.shape), k
        a, b = sd[k].detach().cpu().double().numpy(), v.detach().cpu().double().numpy()
        table = "embedding" in k or k == "linear.weight"
        bad = np.abs(a - b) > rtol * np.abs(b) + max(rtol * float(np.abs(b).max()), 0.0 if table else 5e-6)
        if tower and (table or b.ndim == 2):
            assert bad.mean() <= (table_frac if table else 2e-2), (k, bad.mean())
            assert np.abs(a - b).max() <= 2.2 * 1e-3 * steps, k
        else:
            assert not bad.any(), (k, int(bad.sum()), float(np.abs(a - b).max()))


def _L():
    from rl_ctr_prediction_b200 import _lib
    return _lib


def port_and_model(name, N, F, D, seed=1):
    from rl_ctr_prediction_b200 import pretrain_main as PM
    torch.manual_seed(seed)
    port = TP.make_port(PORT_KIND.get(name, name), N, F, D)
    with torch.no_grad():
        for k, p in port.named_parameters():
            if "embedding" in k or k == "linear.weight":
                p.mul_(0.1)
    if name == "AFM":
        port.dropout_p = 0.0
    port.eval()
    m = PM.get_model(name, N, F, D)
    m.load_state_dict(port.state_dict())
    if name == "AFM":
        m.dropout_p = 0.0
    return port, m.to(DEV).eval()


def batches(N, F, B, steps, seed=0):
    rng = np.random.default_rng(seed)
    return [(torch.as_tensor(rng.integers(0, N, size=(B, F))), torch.as_tensor((rng.random(B) < 0.25).astype(np.int64)))
            for _ in range(steps)]


def freeze_relu_towers(*models):
    for model in models:
        for name in ("mlp", "DN"):
            tower = getattr(model, name, None)
            if tower is not None:
                for p in tower.parameters():
                    p.requires_grad_(False)


# ---- reference-port parity ------------------------------------------------------------------------------------------------------
PARITY = ([(n, 24, 8) for n in NAMES] + [(n, 39, 8) for n in NAMES] +
          [(n, 64, 7 if n == "FFM" else 8) for n in NAMES] +
          [(n, 39, 32) for n in ("FM", "W&D", "DeepFM", "FNN", "IPNN", "OPNN")] +
          [("FFM", 39, 13), ("AFM", 23, 8)])


@pytest.mark.parametrize("mode", ["lazy", "dense"])
@pytest.mark.parametrize("name,F,D", PARITY)
def test_models_match_reference_port(name, F, D, mode, monkeypatch):
    """Three steps of the reference loop body: every pctr and loss, and the final state_dict of all rows, against the CPU port
    trained by torch.optim.Adam (frozen ReLU towers, exact-fp32 tower GEMMs at this batch: tests/test_gpu_latent_dims.py).

    Every model without a tower, and every model's first-step pctr and all its losses, are held to the parity bar.  A tower model's
    table is held to the tower criterion with 2e-3 of the table allowed off the bar (OuterPNN's allowance at F = 15), all inside
    Adam's travel band: at F = 39 and 64 a batch holds 2.6x and 4.3x the row occurrences of F = 15, and the tower's first layer
    takes F*D (+ P) inputs, so more rows sit behind a ReLU that rounding flips.  Measured on a B200: 4.5e-4 .. 8.3e-4 of the table
    for InnerPNN at F = 39, D = 8, FNN at F = 64, D = 8 and W&D at F = 39, D = 32; the other tower models stay under 1e-4."""
    from rl_ctr_prediction_b200 import mlp, optim
    N, B = 50000, 4096
    monkeypatch.setattr(mlp, "FP32_MAX_BATCH", B)
    port, m = port_and_model(name, N, F, D)
    freeze_relu_towers(port, m)
    popt = TP.make_adam(port)
    opt = optim.Adam(params=m.parameters(), lr=1e-3, weight_decay=1e-5, mode=mode)
    lossf = torch.nn.BCELoss()
    for s, (x, y) in enumerate(batches(N, F, B, 3, seed=F + D)):
        y = y.unsqueeze(1)
        with torch.no_grad():
            ref_p = port(x)
        ref_loss = TP.ctr_train_step(port, popt, lossf, x, y)
        p = m(x.to(DEV))
        tl = lossf(p, y.to(DEV).float())
        m.zero_grad()
        tl.backward()
        opt.step()
        close(p, ref_p, rtol=1e-5 if (s == 0 or name not in TOWER) else 1e-3)
        close(tl, ref_loss)
    assert_state(m.state_dict(), port.state_dict(), tower=name in TOWER, table_frac=2e-3)


@pytest.mark.parametrize("F", [24, 39, 64])
def test_afm_past_23_fields_stays_refused(F):
    from rl_ctr_prediction_b200 import pretrain_main as PM
    m = PM.get_model("AFM", 1000, F, 8).to(DEV).eval()
    with pytest.raises(_L().RlctrError, match=r"D <= 32, F <= 23"):
        m(torch.randint(0, 1000, (64, F), device=DEV))


# ---- kernels against fp64 torch -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ip_first", [0, 1])
@pytest.mark.parametrize("F,D", [(23, 1), (23, 32), (24, 1), (24, 7), (24, 32), (39, 7), (39, 32), (64, 1), (64, 7), (64, 32)])
def test_pairdots_against_fp64(F, D, ip_first):
    """rlctr_pairdots_fwd / _bwd at padded pitches against fp64: E copied exactly, ip and the row gradient at the 1e-5 bar, NaN
    pitch pads of every output untouched, and the same bits on a second run."""
    lib = _L().load()
    st = torch.cuda.current_stream().cuda_stream
    B = 1531
    fd, P = F * D, F * (F - 1) // 2
    ld_rows, ld_out, ld_g, ld_gr = fd + 5, fd + P + 3, fd + P + 7, fd + 2
    g = torch.Generator(device=DEV).manual_seed(F * 100 + D)
    rows = torch.full((B, ld_rows), float("nan"), device=DEV)
    rows[:, :fd] = torch.randn(B, fd, device=DEV, generator=g) * 0.5
    gout = torch.full((B, ld_g), float("nan"), device=DEV)
    gout[:, :fd + P] = torch.randn(B, fd + P, device=DEV, generator=g)
    iu = torch.triu_indices(F, F, offset=1, device=DEV)
    e64 = rows[:, :fd].double().contiguous().view(B, F, D).requires_grad_(True)
    ip64 = (e64[:, iu[0]] * e64[:, iu[1]]).sum(2)
    flat = e64.reshape(B, fd)
    ref = torch.cat([ip64, flat], 1) if ip_first else torch.cat([flat, ip64], 1)
    ref.backward(gout[:, :fd + P].double())
    outs = []
    for _ in range(2):
        out = torch.full((B, ld_out), float("nan"), device=DEV)
        grows = torch.full((B, ld_gr), float("nan"), device=DEV)
        assert lib.rlctr_pairdots_fwd(rows.data_ptr(), ld_rows, out.data_ptr(), ld_out, B, F, D, ip_first, st) == 0
        assert lib.rlctr_pairdots_bwd(rows.data_ptr(), ld_rows, gout.data_ptr(), ld_g, grows.data_ptr(), ld_gr, B, F, D, ip_first,
                                      st) == 0
        outs.append((out, grows))
    out, grows = outs[0]
    e_off, ip_off = (P, 0) if ip_first else (0, fd)
    assert torch.equal(out[:, e_off:e_off + fd], rows[:, :fd])
    close(out[:, ip_off:ip_off + P], ip64.detach())
    close(grows[:, :fd], e64.grad.reshape(B, fd))
    assert torch.isnan(out[:, fd + P:]).all() and torch.isnan(grows[:, fd:]).all()
    assert torch.isfinite(out[:, :fd + P]).all() and torch.isfinite(grows[:, :fd]).all()
    for a, b in zip(outs[0], outs[1]):
        assert torch.equal(a.nan_to_num(7.0), b.nan_to_num(7.0))


def _ffm_reference(tab, x, F, D, lin, bias):
    """fp64 logit and the exact partner rows of FFM over the interleaved table (ids outside the table read an all-zero row)."""
    N, rs = tab.shape
    B = x.shape[0]
    ok = (x >= 0) & (x < N)
    r = tab[x.clamp(0, N - 1)] * ok.unsqueeze(2)                                  # [B, F, rs] fp32
    V = r[:, :, :F * D].view(B, F, F, D)                                         # V[b, i, j] = T_j[x_i]
    iu = torch.triu_indices(F, F, offset=1, device=tab.device)
    terms = (V[:, iu[0], iu[1]].double() * V[:, iu[1], iu[0]].double()).sum(2)
    z = bias + r[:, :, lin].double().sum(1) + terms.sum(1)
    scale = r[:, :, lin].double().abs().sum(1) + terms.abs().sum(1) + abs(bias)
    part = torch.zeros(B, F, rs, device=tab.device)
    T = V.transpose(1, 2).clone()                                               # partner row i, block j = T_i[x_j] = V[j, i]
    T[:, torch.arange(F), torch.arange(F)] = 0
    part[:, :, :F * D] = T.reshape(B, F, F * D)
    part[:, :, lin] = 1.0
    return z, scale, part


@pytest.mark.parametrize("F,D,B", [(32, 11, 777), (32, 12, 777), (33, 4, 777), (33, 5, 777), (39, 8, 1531), (39, 13, 1531),
                                   (40, 5, 777), (64, 6, 777), (64, 7, 777), (64, 8, 777), (39, 8, 65536)])
def test_ffm_against_fp64(F, D, B):
    """rlctr_ffm_fwd at every launch variant: the two-warp kernel (F = 32, D = 11), one warp double-buffered (F = 32 at D = 12
    past 200 KB, 33, 39, 40, 64 at D = 6) and single-buffered (F = 64 at D = 7 and 8); even D takes the vectorised partner
    table, odd D the per-element path.  Logits within 1e-5 of the fp64 sum of |terms|, partner rows exact, out-of-range ids
    read zero rows, the same bits on a second run."""
    lib = _L().load()
    st = torch.cuda.current_stream().cuda_stream
    N = 5003
    rs = (F * D + 1 + 3) // 4 * 4
    lin = F * D
    g = torch.Generator(device=DEV).manual_seed(F * 100 + D)
    tab = torch.zeros(N, rs, device=DEV)
    tab[:, :F * D + 1] = torch.randn(N, F * D + 1, device=DEV, generator=g) * 0.2
    x = torch.randint(0, N, (B, F), device=DEV, generator=g)
    x[0, 0] = N + 7
    x[1, F - 1] = -3
    x[2, :] = N
    t = _L().Table(tab.data_ptr(), N, rs, lin, 0, F * D, 0)
    bias = torch.tensor([0.25], device=DEV)
    runs = []
    for _ in range(2):
        logit = torch.empty(B, device=DEV)
        pctr = torch.empty(B, device=DEV)
        part = torch.full((B * F, rs), float("nan"), device=DEV)
        assert lib.rlctr_ffm_fwd(x.data_ptr(), C.byref(t), bias.data_ptr(), logit.data_ptr(), pctr.data_ptr(), 1, part.data_ptr(),
                                 B, F, D, st) == 0
        runs.append((logit, pctr, part))
    logit, pctr, part = runs[0]
    for c0 in range(0, B, 8192):
        c1 = min(B, c0 + 8192)
        z, scale, ref_part = _ffm_reference(tab, x[c0:c1], F, D, lin, 0.25)
        assert bool(((logit[c0:c1].double() - z).abs() <= 1e-5 * scale + 1e-6).all())
        close(pctr[c0:c1], torch.sigmoid(z))
        assert torch.equal(part.view(B, F, rs)[c0:c1], ref_part)
    for a, b in zip(runs[0], runs[1]):
        assert torch.equal(a, b)


# ---- graph and round trip -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,F,D", [("IPNN", 39, 8), ("IPNN", 64, 8), ("FFM", 39, 8), ("FFM", 64, 7)])
def test_graphed_step_equals_eager_and_state_dict_round_trip(name, F, D):
    from rl_ctr_prediction_b200 import graphs, optim
    N, B = 20000, 2048
    lossf = torch.nn.BCELoss()
    _, c = port_and_model(name, N, F, D, seed=7)
    oc = optim.Adam(c.parameters(), lr=1e-3, weight_decay=1e-5)
    gstep = graphs.GraphedTrainStep([(c, oc)], lossf, eager_steps=2)
    _, e = port_and_model(name, N, F, D, seed=7)
    oe = optim.Adam(e.parameters(), lr=1e-3, weight_decay=1e-5)
    for x, y in batches(N, F, B, 5, seed=100 + F):
        x, y = x.to(DEV), y.to(DEV)
        gstep(x, y)
        graphs.eager_step(e, oe, lossf, x, y)
    se, sc = e.state_dict(), c.state_dict()
    for k in se:
        assert torch.equal(se[k], sc[k]), k
    _, f = port_and_model(name, N, F, D, seed=8)
    f.load_state_dict(sc)
    sf = f.state_dict()
    for k in sc:
        assert torch.equal(sf[k], sc[k]), k


# ---- co-located groups ----------------------------------------------------------------------------------------------------------
def _towers(m):
    from rl_ctr_prediction_b200 import mlp
    return [t for t in m.modules() if isinstance(t, mlp.Tower)]


def _group_models(names, N, F, D, seed=3):
    from rl_ctr_prediction_b200 import pretrain_main as PM
    torch.manual_seed(seed)
    ms = [PM.get_model(n, N, F, D).to(DEV).train() for n in names]
    for i, m in enumerate(ms):
        for k, t in enumerate(_towers(m)):
            t.train(True)
            t._rlctr_rng = torch.tensor([1000 * seed + 10 * i + 17 * k, 0], dtype=torch.int64, device=DEV)
    return ms


def _group_batches(N, F, B, steps, seed=11):
    g = torch.Generator().manual_seed(seed)
    per = N // F
    out = []
    for _ in range(steps):
        x = torch.randint(0, per, (B, F), generator=g) + torch.arange(F) * per
        y = (torch.rand(B, generator=g) < 0.3).long()
        out.append((x.to(DEV), y.to(DEV)))
    return out


@pytest.mark.parametrize("mode", ["lazy", "dense"])
@pytest.mark.parametrize("F", [39, 64])
@pytest.mark.parametrize("names,D,max_lines", [(("LR", "FM", "DeepFM"), 8, 1), (("DeepFM", "IPNN"), 10, 1),
                                               (("LR", "FM", "DeepFM"), 16, 2)])
def test_colocated_group_equals_standalone(names, D, max_lines, F, mode):
    """Each member of a co-located group, dropout on, is bit-identical to its stand-alone model (LR within 2e-6: its stand-alone
    forward sums a 1-float row in another order)."""
    from rl_ctr_prediction_b200 import colocated, graphs, optim
    N, B, steps = 3000 if F == 39 else 3008, 512, 4
    sep = _group_models(names, N, F, D)
    grp = [copy.deepcopy(m) for m in sep]
    bs = _group_batches(N, F, B, steps)
    opts = [optim.Adam(m.parameters(), lr=1e-3, weight_decay=1e-5, mode=mode) for m in sep]
    lossf = torch.nn.BCELoss()
    l_sep = np.array([[float(graphs.eager_step(m, o, lossf, x, y)) for m, o in zip(sep, opts)] for x, y in bs])
    group = colocated.colocate(grp, max_lines=max_lines)
    gopt = optim.Adam(group.parameters(), lr=1e-3, weight_decay=1e-5, mode=mode)
    l_grp = np.array([group.train_step(x, y, gopt).cpu().numpy().copy() for x, y in bs])
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
        assert [int(t._rlctr_rng[1]) for t in _towers(sep[i])] == [int(t._rlctr_rng[1]) for t in _towers(grp[i])]


def test_colocated_group_past_its_tile_limit_names_it():
    """DeepFM + InnerPNN at F = 64, D = 14 fit one line, but their tower tiles (2 x 896 floats per sample) exceed the one-line
    gather's 48 KB: the group refuses with that limit."""
    from rl_ctr_prediction_b200 import colocated, optim
    N, F, D = 3008, 64, 14
    group = colocated.colocate(_group_models(("DeepFM", "IPNN"), N, F, D), max_lines=1)
    opt = optim.Adam(group.parameters(), lr=1e-3, weight_decay=1e-5)
    x, y = _group_batches(N, F, 64, 1)[0]
    with pytest.raises(_L().RlctrError, match=r"48 KB"):
        group.train_step(x, y, opt)


# ---- sharded --------------------------------------------------------------------------------------------------------------------
@pytest.fixture
def single_rank_group():
    import torch.distributed as dist
    if not dist.is_initialized():
        import socket
        s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
        dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=0, world_size=1, device_id=torch.device(DEV))
    yield None
    if dist.is_initialized():
        dist.destroy_process_group()


@pytest.mark.parametrize("name", ["IPNN", "FFM"])
def test_sharded_world1_equals_single_gpu(name, single_rank_group):
    from rl_ctr_prediction_b200 import optim, sharded
    N, B, F, D = 20000, 2048, 39, 8
    _, single = port_and_model(name, N, F, D, seed=2)
    s = sharded.ShardedCTR.from_model(single)
    s.eval()
    os_ = optim.Adam(params=s.parameters(), lr=1e-3, weight_decay=1e-5)
    o1 = optim.Adam(params=single.parameters(), lr=1e-3, weight_decay=1e-5)
    lossf = torch.nn.BCELoss()
    for x, y in batches(N, F, B, 3, seed=11):
        x, y = x.to(DEV), y.to(DEV)
        ls = s.train_step(x, y, os_)
        p = single(x)
        l1 = lossf(p, y.reshape(-1, 1).float())
        single.zero_grad()
        l1.backward()
        o1.step()
        close(ls, l1.detach(), rtol=2e-6)
    single.flush()
    rs = single._geom.row_stride
    close(s.gather_table()[:, :rs], single.table.data[:, :rs], rtol=2e-5)


@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("F,D", [(39, 8), (64, 7)])
def test_sharded_ffm_gather_and_update_equal_unsharded(world, F, D):
    """G ranks emulated on one GPU: the FFM forward through peers[] equals the unsharded forward, and the owners' updates through
    the peer-mapped staged partner rows equal one update of the whole table with the concatenated batch -- bit for bit."""
    from rl_ctr_prediction_b200 import sharded
    from rl_ctr_prediction_b200.tables import AdamSchedule
    lib = _L().load()
    st = torch.cuda.current_stream().cuda_stream
    rs, lin, emb, dim = (F * D + 1 + 3) // 4 * 4, F * D, 0, F * D
    N, B = 3001, 200
    rng = np.random.default_rng(world + F)
    full = rng.standard_normal((N, rs)).astype(np.float32) * 0.1
    full[:, lin + 1:] = 0
    ids = rng.integers(0, N, size=(world, B, F))
    sched = AdamSchedule(1e-3, (0.9, 0.999), DEV)
    n_max = sharded.shard_rows(N, world, 0)
    shards = []
    for r in range(world):
        sh = torch.zeros(n_max, rs, device=DEV)
        part = torch.as_tensor(full[r::world]).to(DEV)
        sh[:part.shape[0]] = part
        shards.append(sh)
    tab = torch.as_tensor(full).to(DEV)
    x = torch.as_tensor(ids[1]).to(DEV)
    bias = torch.tensor([0.3], device=DEV)
    outs = []
    for sh_mode in (False, True):
        t = _L().Table(shards[0].data_ptr() if sh_mode else tab.data_ptr(), N, rs, lin, emb, dim, 0)
        if sh_mode:
            t.world = world
            for r in range(world):
                t.peers[r] = shards[r].data_ptr()
        logit = torch.empty(B, device=DEV)
        partners = torch.empty(B * F, rs, device=DEV)
        assert lib.rlctr_ffm_fwd(x.data_ptr(), C.byref(t), bias.data_ptr(), logit.data_ptr(), None, 1, partners.data_ptr(), B, F, D,
                                 st) == 0
        outs.append((logit.clone(), partners.clone()))
    for a, b in zip(*outs):
        assert torch.equal(a, b)

    dl = [torch.as_tensor(rng.standard_normal(B).astype(np.float32) * 0.01).to(DEV) for _ in range(world)]
    srcs = [torch.as_tensor(rng.standard_normal((B * F, rs)).astype(np.float32)).to(DEV) for _ in range(world)]

    def adam(tb):
        m, v = torch.zeros_like(tb), torch.zeros_like(tb)
        step = torch.zeros(1, dtype=torch.int32, device=DEV)
        return _L().Adam(m.data_ptr(), v.data_ptr(), None, _L().ptr(sched.tensor), step.data_ptr(), sched.length, -1, 0.9, 0.999,
                         1e-8, 1e-5), (m, v, step)

    x_all = torch.as_tensor(ids.reshape(-1, F)).to(DEV)
    n = x_all.numel()
    sid = torch.empty(n, dtype=torch.int32, device=DEV)
    ssl = torch.empty_like(sid)
    wsb = lib.rlctr_sort_ws_bytes(n, N)
    ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
    assert lib.rlctr_sort_ids(x_all.data_ptr(), n, N, sid.data_ptr(), ssl.data_ptr(), ws.data_ptr(), wsb, st) == 0
    dl_all, src_all = torch.cat(dl), torch.cat(srcs)
    flags = _L().RLCTR_STAGED_PARTNER
    g = _L().RowGrad(src_all.data_ptr(), dl_all.data_ptr(), None, None, F, flags)
    ref = tab.clone()
    t = _L().Table(ref.data_ptr(), N, rs, lin, emb, dim, 0)
    a, keep = adam(ref)
    rwb = lib.rlctr_rows_ws_bytes(n)
    rws = torch.empty(rwb, dtype=torch.uint8, device=DEV)
    assert lib.rlctr_rows_adam(sid.data_ptr(), ssl.data_ptr(), n, C.byref(g), C.byref(t), C.byref(a), rws.data_ptr(), rwb, st) == 0
    all32 = x_all.reshape(-1).to(torch.int32)
    for rank in range(world):
        n_local = sharded.shard_rows(N, world, rank)
        shard = torch.as_tensor(full[rank::world]).to(DEV).contiguous()
        srows = torch.empty(n, dtype=torch.int32, device=DEV)
        sslots = torch.empty(n, dtype=torch.int32, device=DEV)
        assert lib.rlctr_sort_ids_sharded(all32.data_ptr(), n, world, rank, N, srows.data_ptr(), sslots.data_ptr(), ws.data_ptr(), wsb,
                                          st) == 0
        gs = _L().RowGrad(None, None, None, None, F, flags)
        gs.world, gs.n_per_rank = world, B * F
        for r in range(world):
            gs.peer_dlogit[r] = dl[r].data_ptr()
            gs.peer_staged[r] = srcs[r].data_ptr()
        ts = _L().Table(shard.data_ptr(), n_local, rs, lin, emb, dim, 0)
        as_, keep2 = adam(shard)
        assert lib.rlctr_rows_adam(srows.data_ptr(), sslots.data_ptr(), n, C.byref(gs), C.byref(ts), C.byref(as_), rws.data_ptr(), rwb,
                                   st) == 0
        assert torch.equal(shard, ref[rank::world]), rank
        assert torch.equal(keep2[0], keep[0][rank::world]) and torch.equal(keep2[1], keep[1][rank::world])


# ---- RL side --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("F,D", [(39, 5), (39, 32), (64, 5), (64, 32)])
def test_feature_embedding_against_port(F, D):
    from rl_ctr_prediction_b200.Feature_embedding import Feature_Embedding
    N, B = 50000, 4096
    torch.manual_seed(D)
    port = TP.PortFeatureEmbedding(N, F, D)
    fe = Feature_Embedding(N, F, D)
    fe.load_state_dict(port.state_dict())
    fe = fe.to(DEV)
    x = batches(N, F, B, 1, seed=D)[0][0]
    out = fe(x.to(DEV))
    assert tuple(out.shape) == (B, F * (F - 1) // 2 + F * D)
    close(out, port(x), rtol=1e-5)


def _rl_models(N, F, D):
    from rl_ctr_prediction_b200 import p_model
    from rl_ctr_prediction_b200.Feature_embedding import Feature_Embedding
    models = {0: p_model.LR(N), 1: p_model.FM(N, D), 2: p_model.FFM(N, F, D)}
    for m in models.values():
        with torch.no_grad():
            m.table.mul_(0.1)
        m.to(DEV).eval()
    fe = Feature_Embedding(N, F, D).to(DEV)
    fe.load_embedding(models[1].state_dict())
    return models, fe


def test_all_main_train_step_at_39_fields():
    from rl_ctr_prediction_b200 import all_main
    torch.manual_seed(3)
    N, F, D, B, M = 5000, 39, 5, 512, 3
    models, fe = _rl_models(N, F, D)
    assert fe.forward(torch.randint(0, N, (4, F), device=DEV)).shape[1] == F * (F - 1) // 2 + F * D
    ddqn, ddpg = all_main.get_model(M, N, F, D, 128, 4096, DEV, "1458")
    rng = np.random.default_rng(0)
    for _ in range(2):
        x = torch.as_tensor(rng.integers(0, N, size=(B, F))).to(DEV)
        y = torch.as_tensor((rng.random((B, 1)) < 0.3).astype(np.int64)).to(DEV)
        y_preds, rewards, td, al = all_main.train_step(ddqn, ddpg, models, x, y, fe, 0.5, DEV)
        assert y_preds.shape == (B, 1) and rewards.shape == (B, 1)
        assert torch.isfinite(y_preds).all() and np.isfinite(td) and np.isfinite(al)
    assert torch.equal(ddqn.memory[B:2 * B, :F].long(), x)


def test_td3_v10_train_step_at_39_fields():
    from rl_ctr_prediction_b200 import hybrid_td3_main_per_v10 as V10, v10_Hybrid_TD3_model_PER as T
    torch.manual_seed(5)
    N, F, D, B, M = 5000, 39, 5, 384, 3
    models, fe = _rl_models(N, F, D)
    agent = T.Hybrid_TD3_Model(N, F, D, M, memory_size=4 * B, batch_size=64, device=DEV)
    assert agent.input_dims == F * (F - 1) // 2 + F * D
    rng = np.random.default_rng(1)
    for index in (0, 1000):
        x = torch.as_tensor(rng.integers(0, N, size=(B, F))).to(DEV)
        y = torch.as_tensor((rng.random((B, 1)) < 0.3).astype(np.int64)).to(DEV)
        y_preds, rewards, critic_loss = V10.train_step(agent, models, x, y, fe, index, DEV)
        assert torch.isfinite(y_preds).all() and torch.isfinite(rewards).all()
        assert (critic_loss is None) == (index < V10.RANDOM_STEPS)
        if critic_loss is not None:
            assert np.isfinite(float(critic_loss))


# ---- end to end -----------------------------------------------------------------------------------------------------------------
def test_pretrain_main_at_39_fields(tmp_path):
    """pretrain_main.main on a synthetic 39-field set: FM, then IPNN from FM's FMbest.pth embedding, then FFM at D = 8."""
    import os
    from rl_ctr_prediction_b200 import pretrain_main as PM
    F, D = 39, 8
    rng = np.random.default_rng(0)
    root = str(tmp_path) + "/"
    os.makedirs(root + "cretio/1458/")
    n = 600
    ids = np.stack([rng.integers(f * 20, f * 20 + 20, size=n) for f in range(F)], axis=1)
    rows = np.column_stack([(rng.random(n) < 0.3).astype(np.int64), ids])
    np.savetxt(root + "cretio/1458/train.txt", rows, fmt="%d", delimiter=",")
    np.savetxt(root + "cretio/1458/day_index.csv", np.array([[6, 0, 199], [11, 200, 399], [12, 400, 599]]), fmt="%d", delimiter=",")
    os.makedirs(root + "params/")
    feature_nums = PM.get_dataset(root, "cretio/", "1458/", 11, 12)[-1]
    for name in ("FM", "IPNN", "FFM"):
        PM.setup_seed(1)
        PM.main(data_path=root, dataset_name="cretio/", campaign_id="1458/", valid_day=11, test_day=12, latent_dims=D,
                model_name=name, epoch=2, learning_rate=1e-3, weight_decay=1e-5, early_stop_type="loss", batch_size=128, device=DEV,
                save_param_dir=root + "params/")
        sd = torch.load(root + f"params/1458/{name}best.pth")
        port = TP.make_port(PORT_KIND.get(name, name), feature_nums, F, D)
        ref = port.state_dict()
        assert set(sd) == set(ref), name
        for k in ref:
            assert tuple(sd[k].shape) == tuple(ref[k].shape), (name, k)
        assert all(torch.isfinite(v).all() for v in sd.values())
