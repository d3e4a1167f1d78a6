"""Every get_model name at latent sizes past the ones the library first served: D in {5, 16, 20, 32} at F = 15.

D = 5 and 20 reach the AFM kernels for D other than 4, 8 and 10 (per-lane backward for D <= 10, the lane-per-unit kernels
above), D = 20 and 32 the 16-column DCN cross network (F*D > 256) and the FFM row update with four chunks per lane (rows over
256 floats), D = 32 the 36-float FM-type rows (a first-order column plus 32 latent floats) in the gather and the update."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import torch_port as TP

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
F = 15
DIMS = [5, 16, 20, 32]
NAMES = ["LR", "FM", "FFM", "W&D", "DeepFM", "FNN", "IPNN", "OPNN", "DCN", "AFM"]
PORT_KIND = {"W&D": "WideAndDeep", "IPNN": "InnerPNN", "OPNN": "OuterPNN"}


def close(a, b, rtol=1e-5, atol=None):
    """|a - b| <= rtol * max(|b|, scale of b) (tests/test_gpu_models.py's bar)."""
    a = a.detach().cpu().double().numpy() if isinstance(a, torch.Tensor) else np.asarray(a, np.float64)
    b = b.detach().cpu().double().numpy() if isinstance(b, torch.Tensor) else np.asarray(b, np.float64)
    if atol is None:
        atol = rtol * (np.abs(b).max() if b.size else 0.0)
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol)


TOWER = {"W&D", "DeepFM", "FNN", "IPNN", "OPNN", "DCN"}


def assert_state(sd, ref_sd, tower=False, steps=3, rtol=2e-5, table_frac=1e-4):
    """Every parameter at the parity bar.  Models with a tower (tests/test_gpu_parity_scale.py's argument): where the gradient a
    tower hands back is rounding-level noise, Adam's step is +-lr in a noise-determined direction in the reference too, so two
    correct fp32 GEMMs disagree on a few elements -- all of them inside Adam's travel band (`steps` steps of lr)."""
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


def port_and_model(name, N, D, seed=1):
    """A CPU port of the reference model and the library model loaded from the port's state_dict (tables scaled by 0.1 so the
    sigmoid does not saturate)."""
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


def batches(N, B, steps, seed=0):
    rng = np.random.default_rng(seed)
    return [(torch.as_tensor(rng.integers(0, N, size=(B, F))), torch.as_tensor((rng.random(B) < 0.25).astype(np.int64)))
            for _ in range(steps)]


def freeze_relu_towers(*models):
    """Take the ReLU towers' weights (``mlp``; DCN's deep net ``DN``) out of training on both sides.  They still run forward and
    hand their gradient back to the rows; only their own Adam step is skipped."""
    for model in models:
        for name in ("mlp", "DN"):
            tower = getattr(model, name, None)
            if tower is not None:
                for p in tower.parameters():
                    p.requires_grad_(False)


@pytest.mark.parametrize("mode", ["lazy", "dense"])
@pytest.mark.parametrize("D", DIMS)
@pytest.mark.parametrize("name", NAMES)
def test_models_match_reference_port(name, D, mode, monkeypatch):
    """Three steps of the reference loop body: every pctr and loss, and the final state_dict of all rows, against the CPU port
    trained by torch.optim.Adam.

    The towers take the exact-fp32 GEMM at this batch, and their weights are frozen on both sides: a tower weight whose gradient
    cancels to rounding level takes Adam's +-lr step in a direction set by that rounding (in the reference too), flips ReLUs
    near zero in the next step and moves the rows behind them by up to lr -- up to 0.2 % of the table at this batch.  Frozen
    towers still run forward and hand their gradient back to the rows.  What remains for a tower model is the smaller form of
    the same effect through the rows themselves, so it is held to tests/test_gpu_parity_scale.py's tower criterion: after the
    first step pctr within 1e-3 of the scale, table elements off the bar on at most 1e-4 of the table and all inside Adam's
    travel band.  OuterPNN feeds its tower D * (sum_f v_f)^2 (about 5 at D = 32), so its first layer's pre-activations are large
    and its ReLUs flip more often: its table is allowed 2e-3 off the bar, inside the band.  The unchanged parent library gives
    the same OuterPNN numbers bit for bit at D = 16 and 32, which need no kernel this size selects anew.  Every model without a
    tower, and every model's first step and losses, are held to the parity bar."""
    from rl_ctr_prediction_b200 import mlp, optim
    N, B = 50000, 4096
    monkeypatch.setattr(mlp, "FP32_MAX_BATCH", B)
    port, m = port_and_model(name, N, D)
    freeze_relu_towers(port, m)
    popt = TP.make_adam(port)
    opt = optim.Adam(params=m.parameters(), lr=1e-3, weight_decay=1e-5, mode=mode)
    lossf = torch.nn.BCELoss()
    for s, (x, y) in enumerate(batches(N, B, 3, seed=D)):
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
    assert_state(m.state_dict(), port.state_dict(), tower=name in TOWER, table_frac=2e-3 if name == "OPNN" else 1e-4)


def _afm_torch(rows, packed, Ft, Dt, masks):
    Bt = rows.shape[0]
    npair = Ft * (Ft - 1) // 2
    o = 0
    Wa = packed[o:o + Dt * Dt].view(Dt, Dt); o += Dt * Dt
    ba = packed[o:o + Dt]; o += Dt
    ws = packed[o:o + Dt]; o += Dt
    bs = packed[o]; o += 1
    fcw = packed[o:o + Dt]; o += Dt
    fcb = packed[o]
    e = rows.view(Bt, Ft, Dt)
    idx = torch.triu_indices(Ft, Ft, offset=1)
    ip = e[:, idx[0]] * e[:, idx[1]]
    a = torch.relu(ip @ Wa.t() + ba)
    s = a @ ws + bs
    sc = torch.softmax(s, dim=1) * masks[:, :npair]
    attn = (sc.unsqueeze(2) * ip).sum(dim=1) * masks[:, npair:]
    return (attn @ fcw + fcb).unsqueeze(1)


@pytest.mark.parametrize("Ft,Dt", [(15, 1), (15, 5), (15, 11), (15, 16), (15, 20), (15, 32), (23, 32)])
def test_afm_kernels_against_torch_fp64(Ft, Dt):
    """rlctr_afm_fwd / _bwd at the new D against the reference expression in fp64 autograd: given masks, hash masks regenerated
    by the backward, ragged batch, padded pitch; bit-identical from run to run."""
    from rl_ctr_prediction_b200 import p_model
    torch.manual_seed(Dt)
    Bt = 1531
    npair = Ft * (Ft - 1) // 2
    pitch = (Ft * Dt + 3) // 4 * 4 + 4
    buf = torch.full((Bt, pitch), float("nan"), device=DEV)
    buf[:, :Ft * Dt] = torch.randn(Bt, Ft * Dt, device=DEV) * 0.7
    rows = buf[:, :Ft * Dt].requires_grad_(True)
    packed = (torch.randn(Dt * Dt + 3 * Dt + 2, device=DEV) * (0.4 if Dt <= 10 else 1.2 / Dt ** 0.5)).requires_grad_(True)
    masks = (torch.rand(Bt, npair + Dt, device=DEV) >= 0.2).float() / 0.8
    g = torch.randn(Bt, 1, device=DEV)
    for mk in (masks, None):
        rows.grad = packed.grad = None
        y = p_model._AFMAttention.apply(rows, packed, Ft, Dt, 0.2 if mk is not None else 0.0, None, mk)
        y.backward(g)
        r64 = buf[:, :Ft * Dt].detach().double().requires_grad_(True)
        p64 = packed.detach().double().requires_grad_(True)
        m64 = mk.double() if mk is not None else torch.ones(Bt, npair + Dt, device=DEV, dtype=torch.float64)
        ref = _afm_torch(r64, p64, Ft, Dt, m64)
        ref.backward(g.double())
        close(y, ref.detach(), rtol=1e-5)
        close(rows.grad, r64.grad, rtol=1e-5)
        close(packed.grad, p64.grad, rtol=1e-5)
    y2 = p_model._AFMAttention.apply(rows, packed, Ft, Dt, 0.0, None, None)
    pg = packed.grad.clone()
    rows.grad = packed.grad = None
    y2.backward(g)
    assert torch.equal(y2, y) and torch.equal(packed.grad, pg)
    # hash-drawn masks: the counter moves by B * (P + D), the same snapshot draws the same output, and the backward (which
    # regenerates the masks from the snapshot) gives d y / d fc_b = sum g whatever the masks
    rng = torch.tensor([987654321, 0], dtype=torch.int64, device=DEV)
    rows.grad = packed.grad = None
    yh = p_model._AFMAttention.apply(rows, packed, Ft, Dt, 0.2, rng, None)
    yh.backward(g)
    assert int(rng[1].item()) == Bt * (npair + Dt)
    assert torch.equal(yh, p_model._AFMAttention.apply(rows, packed, Ft, Dt, 0.2, torch.tensor([987654321, 0], dtype=torch.int64,
                                                                                             device=DEV), None))
    assert torch.isfinite(rows.grad).all() and torch.isfinite(packed.grad).all()
    close(packed.grad[-1], g.sum())


@pytest.mark.parametrize("fd", [270, 300, 480, 512])
def test_cross_kernels_against_torch_fp64(fd):
    """rlctr_cross_fwd / _bwd at F*D over 256 (16 columns per lane) against fp64 autograd; bit-identical from run to run."""
    from rl_ctr_prediction_b200 import p_model
    torch.manual_seed(fd)
    Bt, L = 2077, 5
    buf = torch.full((Bt, fd + 4), float("nan"), device=DEV)
    buf[:, :fd] = torch.randn(Bt, fd, device=DEV) * 0.3
    rows = buf[:, :fd].requires_grad_(True)
    W = (torch.randn(L, fd, device=DEV) * 0.05).requires_grad_(True)
    Bv = (torch.randn(L, fd, device=DEV) * 0.1).requires_grad_(True)
    g = torch.randn(Bt, fd, device=DEV)
    out = p_model._CrossNet.apply(rows, W, Bv)
    out.backward(g)
    r64, W64, B64 = (t.detach().double().requires_grad_(True) for t in (buf[:, :fd], W, Bv))
    xl = r64
    for l in range(L):
        xl = r64 * (xl @ W64[l]).unsqueeze(1) + B64[l] + xl
    xl.backward(g.double())
    close(out, xl.detach(), rtol=1e-5)
    close(rows.grad, r64.grad, rtol=1e-5)
    close(W.grad, W64.grad, rtol=1e-5)
    close(Bv.grad, B64.grad, rtol=1e-5)
    gw, gr = W.grad.clone(), rows.grad.clone()
    W.grad = Bv.grad = rows.grad = None
    out2 = p_model._CrossNet.apply(rows, W, Bv)
    out2.backward(g)
    assert torch.equal(out, out2) and torch.equal(W.grad, gw) and torch.equal(rows.grad, gr)


@pytest.mark.parametrize("fm", [0, 1])
def test_36_float_gather_against_torch(fm):
    """rlctr_embed_fwd on 36-float rows ([w, v_0..v_31, pad]): logit / pctr, the column sums and the tower rows against fp64,
    and the FM-term row gradient (rowgrad_combine with the saved sums) of the update at that width against autograd."""
    lib = _L().load()
    N, B, D, rs = 7001, 777, 32, 36
    rng = np.random.default_rng(36 + fm)
    tab = np.zeros((N, rs), np.float32)
    tab[:, :1 + D] = rng.standard_normal((N, 1 + D)).astype(np.float32) * 0.2
    x = rng.integers(0, N, size=(B, F))
    x[0, 0] = N + 3                                       # out of range: an all-zero row
    td = torch.as_tensor(tab).to(DEV)
    t = _L().Table(td.data_ptr(), N, rs, 0, 1, D, 0)
    bias = torch.tensor([0.1], device=DEV)
    logit = torch.empty(B, device=DEV)
    pctr = torch.empty(B, device=DEV)
    sums = torch.empty(B, rs, device=DEV)
    pitch = F * D + 4
    rows = torch.full((B, pitch), float("nan"), device=DEV)
    xd = torch.as_tensor(x).to(DEV)
    st = torch.cuda.current_stream().cuda_stream
    assert lib.rlctr_embed_fwd(xd.data_ptr(), C.byref(t), bias.data_ptr(), logit.data_ptr(), pctr.data_ptr(), 1, sums.data_ptr(),
                               rows.data_ptr(), pitch, B, F, _L().RLCTR_FM_TERM if fm else 0, st) == 0
    e = np.zeros((B, F, rs))
    ok = x < N
    e[ok] = tab[x[ok]].astype(np.float64)
    S = e.sum(axis=1)
    z = 0.1 + S[:, 0]
    if fm:
        v = e[:, :, 1:1 + D]
        z = z + 0.5 * (v.sum(axis=1) ** 2 - (v ** 2).sum(axis=1)).sum(axis=1)
    close(logit, z)
    close(pctr, 1 / (1 + np.exp(-z)))
    close(sums, S)
    assert torch.equal(rows[:, :F * D].cpu(), torch.as_tensor(e[:, :, 1:1 + D].reshape(B, F * D), dtype=torch.float32))
    # the FM-term gradient at this width: rows_grad_dense(dlogit, sums) == d logit / d row by autograd, per id
    if fm:
        dl = torch.as_tensor(rng.standard_normal(B).astype(np.float32)).to(DEV)
        sid = torch.empty(B * F, dtype=torch.int32, device=DEV)
        ssl = torch.empty_like(sid)
        wsb = lib.rlctr_sort_ws_bytes(B * F, N)
        ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
        assert lib.rlctr_sort_ids(xd.data_ptr(), B * F, N, sid.data_ptr(), ssl.data_ptr(), ws.data_ptr(), wsb, st) == 0
        grad = _L().RowGrad(None, dl.data_ptr(), sums.data_ptr(), None, F, 0)
        dense = torch.zeros(N, rs, device=DEV)
        rwb = lib.rlctr_rows_ws_bytes(B * F)
        rws = torch.empty(rwb, dtype=torch.uint8, device=DEV)
        assert lib.rlctr_rows_grad_dense(sid.data_ptr(), ssl.data_ptr(), B * F, C.byref(grad), C.byref(t), dense.data_ptr(),
                                         rws.data_ptr(), rwb, st) == 0
        T = torch.as_tensor(tab, dtype=torch.float64).requires_grad_(True)
        xc = torch.as_tensor(np.where(ok, x, 0))
        ee = T[xc] * torch.as_tensor(ok, dtype=torch.float64).unsqueeze(2)
        w1, vv = ee[:, :, 0], ee[:, :, 1:1 + D]
        zz = w1.sum(1) + 0.5 * (vv.sum(1) ** 2 - (vv ** 2).sum(1)).sum(1)
        (zz * dl.cpu().double()).sum().backward()
        close(dense[:, :1 + D], T.grad[:, :1 + D])
        assert float(dense[:, 1 + D:].abs().max()) == 0.0


@pytest.mark.parametrize("name", ["FM", "FFM", "DCN", "AFM"])
def test_large_batch_d32(name):
    """B = 65536 at D = 32: grid-capped forward / backward kernels and heavy rows (Zipf ids), against the port (one step)."""
    from rl_ctr_prediction_b200 import optim
    N, B, D = 20000, 65536, 32
    port, m = port_and_model(name, N, D, seed=4)
    popt = TP.make_adam(port)
    opt = optim.Adam(params=m.parameters(), lr=1e-3, weight_decay=1e-5)
    rng = np.random.default_rng(9)
    x = torch.as_tensor(np.minimum(rng.zipf(1.3, size=(B, F)) - 1, N - 1))
    y = torch.as_tensor((rng.random(B) < 0.25).astype(np.int64)).unsqueeze(1)
    lossf = torch.nn.BCELoss()
    with torch.no_grad():
        ref_p = port(x)
    ref_loss = TP.ctr_train_step(port, popt, lossf, x, y)
    p = m(x.to(DEV))
    tl = lossf(p, y.to(DEV).float())
    m.zero_grad()
    tl.backward()
    opt.step()
    close(p, ref_p)
    close(tl, ref_loss)
    assert_state(m.state_dict(), port.state_dict(), tower=name in TOWER, steps=1, rtol=5e-5)


@pytest.mark.parametrize("D", [5, 32])
@pytest.mark.parametrize("name", NAMES)
def test_bit_identity(name, D):
    """At the new D: the fused step gives the autograd loop body's losses and parameters, the graphed step equals the eager step
    bit for bit, and the state_dict round-trips bit for bit."""
    from rl_ctr_prediction_b200 import graphs, optim, pretrain_main as PM
    N, B = 20000, 2048
    a, b, c = (port_and_model(name, N, D, seed=7)[1] for _ in range(3))
    oa = optim.Adam(a.parameters(), lr=1e-3, weight_decay=1e-5)
    ob = optim.Adam(b.parameters(), lr=1e-3, weight_decay=1e-5)
    oc = optim.Adam(c.parameters(), lr=1e-3, weight_decay=1e-5)
    lossf = torch.nn.BCELoss()
    gstep = graphs.GraphedTrainStep([(c, oc)], lossf, eager_steps=2)
    for x, y in batches(N, B, 5, seed=100 + D):
        x, y = x.to(DEV), y.to(DEV)
        la = PM.fused_train_step(a, oa, x, y)
        p = b(x)
        lb = lossf(p, y.reshape(-1, 1).float())
        b.zero_grad()
        lb.backward()
        ob.step()
        close(la, lb.detach(), rtol=2e-6)
        gstep(x, y)
    sa, sb = a.state_dict(), b.state_dict()
    for k in sb:
        close(sa[k], sb[k], rtol=2e-5, atol=max(2e-5 * float(sb[k].abs().max()), 5e-6))
    # graphed == eager, bit for bit: replay a fresh copy eagerly with graphs.eager_step over the same batches
    _, e = port_and_model(name, N, D, seed=7)
    oe = optim.Adam(e.parameters(), lr=1e-3, weight_decay=1e-5)
    for x, y in batches(N, B, 5, seed=100 + D):
        graphs.eager_step(e, oe, lossf, x.to(DEV), y.to(DEV))
    se, sc = e.state_dict(), c.state_dict()
    for k in se:
        assert torch.equal(se[k], sc[k]), k
    # state_dict round trip
    _, f = port_and_model(name, N, D, seed=8)
    f.load_state_dict(sc)
    sf = f.state_dict()
    for k in sc:
        assert torch.equal(sf[k], sc[k]), k


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


@pytest.mark.parametrize("name", NAMES)
def test_sharded_world1_equals_single_gpu_d32(name, single_rank_group):
    """World-1 ShardedCTR.from_model at D = 32 takes the single-GPU model's steps: its fused loss head against the autograd loop
    body, at the parity bar."""
    from rl_ctr_prediction_b200 import optim, sharded
    N, B, D = 20000, 2048, 32
    _, single = port_and_model(name, N, D, seed=2)
    s = sharded.ShardedCTR.from_model(single)
    s.eval()
    os_ = optim.Adam(params=s.parameters(), lr=1e-3, weight_decay=1e-5)
    o1 = optim.Adam(params=single.parameters(), lr=1e-3, weight_decay=1e-5)
    lossf = torch.nn.BCELoss()
    for x, y in batches(N, B, 3, seed=11):
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
@pytest.mark.parametrize("kind", ["fm36", "ffm484"])
def test_sharded_gather_and_update_equal_unsharded(world, kind):
    """G ranks emulated on one GPU at the new widths: the gather through peers[] equals the unsharded gather, and the owners'
    updates (FM-term rows through the sums, FFM through the peer-mapped staged partner rows) equal one update of the whole
    table with the concatenated batch -- bit for bit."""
    from rl_ctr_prediction_b200 import sharded
    from rl_ctr_prediction_b200.tables import AdamSchedule
    lib = _L().load()
    st = torch.cuda.current_stream().cuda_stream
    D = 32
    if kind == "fm36":
        rs, lin, emb, dim = 36, 0, 1, D
    else:
        rs, lin, emb, dim = 484, F * D, 0, F * D
    N, B = 3001, 200
    rng = np.random.default_rng(world)
    full = rng.standard_normal((N, rs)).astype(np.float32) * 0.1
    full[:, max(lin, emb + dim - 1) + 1:] = 0
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
    # ---- forward: one rank's batch through peers[] == the unsharded table
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
        if kind == "fm36":
            sums = torch.empty(B, rs, device=DEV)
            rows = torch.empty(B, F * D, device=DEV)
            assert lib.rlctr_embed_fwd(x.data_ptr(), C.byref(t), bias.data_ptr(), logit.data_ptr(), None, 1, sums.data_ptr(),
                                       rows.data_ptr(), 0, B, F, 1, st) == 0
            outs.append((logit.clone(), sums.clone(), rows.clone()))
        else:
            partners = torch.empty(B * F, rs, device=DEV)
            assert lib.rlctr_ffm_fwd(x.data_ptr(), C.byref(t), bias.data_ptr(), logit.data_ptr(), None, 1, partners.data_ptr(), B, F,
                                     D, st) == 0
            outs.append((logit.clone(), partners.clone()))
    for a, b in zip(*outs):
        assert torch.equal(a, b)

    # ---- update: owners with peer-mapped gradient sources == one table, concatenated batch
    dl = [torch.as_tensor(rng.standard_normal(B).astype(np.float32) * 0.01).to(DEV) for _ in range(world)]
    if kind == "fm36":
        srcs = [torch.as_tensor(rng.standard_normal((B, rs)).astype(np.float32)).to(DEV) for _ in range(world)]
    else:
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
    flags = 0 if kind == "fm36" else _L().RLCTR_STAGED_PARTNER
    if kind == "fm36":
        g = _L().RowGrad(None, dl_all.data_ptr(), src_all.data_ptr(), None, F, flags)
    else:
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
            if kind == "fm36":
                gs.peer_sums[r] = srcs[r].data_ptr()
            else:
                gs.peer_staged[r] = srcs[r].data_ptr()
        ts = _L().Table(shard.data_ptr(), n_local, rs, lin, emb, dim, 0)
        as_, keep2 = adam(shard)
        assert lib.rlctr_rows_adam(srows.data_ptr(), sslots.data_ptr(), n, C.byref(gs), C.byref(ts), C.byref(as_), rws.data_ptr(), rwb,
                                   st) == 0
        assert torch.equal(shard, ref[rank::world]), rank
        assert torch.equal(keep2[0], keep[0][rank::world]) and torch.equal(keep2[1], keep[1][rank::world])


@pytest.mark.parametrize("D", [5, 32])
def test_feature_embedding_against_port(D):
    from rl_ctr_prediction_b200.Feature_embedding import Feature_Embedding
    N, B = 50000, 4096
    torch.manual_seed(D)
    port = TP.PortFeatureEmbedding(N, F, D)
    fe = Feature_Embedding(N, F, D)
    fe.load_state_dict(port.state_dict())
    fe = fe.to(DEV)
    x = batches(N, B, 1, seed=D)[0][0]
    close(fe(x.to(DEV)), port(x), rtol=1e-5)


def test_pretrain_main_afm_d32(tmp_path):
    """python -m rl_ctr_prediction_b200.pretrain_main --latent_dims 32 --model_name AFM, end to end on a small synthetic set."""
    import os
    from rl_ctr_prediction_b200 import pretrain_main as PM
    rng = np.random.default_rng(0)
    root = str(tmp_path) + "/"
    os.makedirs(root + "ipinyou/1458/")
    n = 600
    ids = np.stack([rng.integers(f * 20, f * 20 + 20, size=n) for f in range(F)], axis=1)
    rows = np.column_stack([(rng.random(n) < 0.3).astype(np.int64), ids])
    np.savetxt(root + "ipinyou/1458/train.txt", rows, fmt="%d", delimiter=",")
    np.savetxt(root + "ipinyou/1458/day_index.csv", np.array([[6, 0, 199], [11, 200, 399], [12, 400, 599]]), fmt="%d", delimiter=",")
    os.makedirs(root + "params/")
    PM.setup_seed(1)
    PM.main(data_path=root, dataset_name="ipinyou/", campaign_id="1458/", valid_day=11, test_day=12, latent_dims=32,
            model_name="AFM", epoch=2, learning_rate=1e-3, weight_decay=1e-5, early_stop_type="loss", batch_size=128, device=DEV,
            save_param_dir=root + "params/")
    sd = torch.load(root + "params/1458/AFMbest.pth")
    assert tuple(sd["feature_embedding.weight"].shape)[1] == 32 and tuple(sd["attention_net.weight"].shape) == (32, 32)
    assert all(torch.isfinite(v).all() for v in sd.values())
