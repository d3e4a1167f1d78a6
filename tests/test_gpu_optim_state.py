"""Resumable training: optim.Adam / optim.Adagrad ``state_dict()`` / ``load_state_dict()`` and torch's LR schedulers.

Bit for bit against our own uninterrupted run (``torch.equal`` on losses, ``model.state_dict()`` and ``opt.state_dict()``): a run
trains k steps, saves model and optimizer through ``torch.save``, and a fresh model and optimizer loaded with
``torch.load(map_location="cpu")`` train m more -- for all ten models, the three load orders, co-located groups, the row-sharded
models at world 1 and graphed steps (including a load whose step is past the schedule a captured graph holds).  The source run
keeps training after its ``state_dict()`` calls: it must equal a run that never made them.  Against stock torch on the CPU port
(oracle/torch_port.py), at the bars of test_gpu_optim.py / test_gpu_adagrad.py: resume through torch's own state_dict, every
listed LR scheduler (its state resumed too), and dense-only checkpoints exchanged with torch.optim both ways."""
import copy
import io

import numpy as np
import pytest
import torch
from torch.optim import lr_scheduler as S

from oracle import torch_port as TP

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NAMES = ["LR", "FM", "FFM", "DeepFM", "W&D", "FNN", "IPNN", "OPNN", "DCN", "AFM"]
SETTINGS = {"adam_lazy": ("Adam", dict(lr=1e-2, weight_decay=1e-5)),
            "adam_dense": ("Adam", dict(lr=1e-2, weight_decay=1e-5, mode="dense")),
            "adam_sparse": ("Adam", dict(lr=1e-2, weight_decay=1e-5, mode="sparse")),
            "adagrad_wd0": ("Adagrad", dict(lr=1e-2)),
            "adagrad_wd": ("Adagrad", dict(lr=1e-2, weight_decay=1e-4))}
ORDERS = ("model_build_opt", "build_model_opt", "build_opt_model")


def _opt(setting, params):
    from rl_ctr_prediction_b200 import optim
    cls, kw = SETTINGS[setting]
    return getattr(optim, cls)(params, **kw)


def _model(name, N, F, D, seed):
    from rl_ctr_prediction_b200 import pretrain_main as PM
    torch.manual_seed(seed)
    m = PM.get_model(name, N, F, D).to(DEV).eval()           # towers without dropout: the model's RNG is not optimizer state
    if hasattr(m, "dropout_p"):
        m.dropout_p = 0.0
    return m


def _batches(N, F, steps, B=128, seed=0):
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(steps):
        x = (torch.rand(B, F, generator=g) ** 4 * N).long().clamp_(0, N - 1)     # skewed: some rows skip steps (lazy replay)
        out.append((x.to(DEV), (torch.rand(B, 1, generator=g) < 0.3).long().to(DEV)))
    return out


def _eager(m, opt, x, y):
    from rl_ctr_prediction_b200 import graphs
    return float(graphs.eager_step(m, opt, torch.nn.BCELoss(), x, y))


def _save(model, opt):
    buf = io.BytesIO()
    torch.save({"model": model.state_dict(), "opt": opt.state_dict()}, buf)
    buf.seek(0)
    return torch.load(buf, map_location="cpu", weights_only=False)


def _restore(make, make_opt, ck, order):
    """A fresh model (other initial values) and optimizer, loaded from ``ck`` in ``order``."""
    m = make(seed=99)
    if order == "model_build_opt":
        m.load_state_dict(ck["model"])
        o = make_opt(m)
        o.load_state_dict(ck["opt"])
    elif order == "build_model_opt":
        o = make_opt(m)
        m.load_state_dict(ck["model"])
        o.load_state_dict(ck["opt"])
    else:
        o = make_opt(m)
        o.load_state_dict(ck["opt"])
        m.load_state_dict(ck["model"])
    return m, o


def assert_sd_equal(a, b, where=""):
    """Equal nested state (dicts, lists, tensors, numbers) bit for bit."""
    if isinstance(a, dict):
        assert a.keys() == b.keys(), (where, a.keys(), b.keys())
        for k in a:
            assert_sd_equal(a[k], b[k], f"{where}.{k}")
    elif isinstance(a, (list, tuple)):
        assert len(a) == len(b), where
        for i, (u, v) in enumerate(zip(a, b)):
            assert_sd_equal(u, v, f"{where}[{i}]")
    elif isinstance(a, torch.Tensor):
        assert isinstance(b, torch.Tensor) and a.dtype == b.dtype and a.shape == b.shape, where
        assert torch.equal(a.cpu(), b.cpu()), where
    else:
        assert a == b, (where, a, b)


def _resume_case(make, make_opt, step_fn, batches, k, order="build_model_opt"):
    """Uninterrupted run A against: run B, which saves at step k (and calls opt.state_dict() again after one more step) and
    keeps going, and run C, restored from B's checkpoint.  All three must end with the same bits."""
    a = make(seed=1)
    oa = make_opt(a)
    la = [step_fn(a, oa, x, y) for x, y in batches]
    b = make(seed=1)
    ob = make_opt(b)
    lb = [step_fn(b, ob, x, y) for x, y in batches[:k]]
    ck = _save(b, ob)
    lb.append(step_fn(b, ob, *batches[k]))
    ob.state_dict()                                           # a mid-run export changes nothing either
    lb += [step_fn(b, ob, x, y) for x, y in batches[k + 1:]]
    c, oc = _restore(make, make_opt, ck, order)
    lc = la[:k] + [step_fn(c, oc, x, y) for x, y in batches[k:]]
    assert la == lb and la == lc, (la, lb, lc)
    sa = (a.state_dict(), oa.state_dict())
    assert_sd_equal(sa, (b.state_dict(), ob.state_dict()), "uninterrupted vs mid-run exports")
    assert_sd_equal(sa, (c.state_dict(), oc.state_dict()), "uninterrupted vs resumed")
    return a, oa, c, oc


@pytest.mark.parametrize("setting", list(SETTINGS))
@pytest.mark.parametrize("name", NAMES)
def test_resume_equals_uninterrupted(name, setting):
    N, F, D = 400, 15, 10
    _resume_case(lambda seed: _model(name, N, F, D, seed), lambda m: _opt(setting, m.parameters()), _eager,
                 _batches(N, F, 7), 3)


@pytest.mark.parametrize("order", ORDERS)
@pytest.mark.parametrize("setting", ["adam_lazy", "adagrad_wd"])
@pytest.mark.parametrize("name", ["FM", "DeepFM", "FFM"])
def test_load_orders(name, setting, order):
    N, F, D = 400, 15, 10
    _resume_case(lambda seed: _model(name, N, F, D, seed), lambda m: _opt(setting, m.parameters()), _eager,
                 _batches(N, F, 6, seed=5), 2, order=order)


@pytest.mark.parametrize("setting", ["adam_lazy", "adagrad_wd"])
def test_ffm_separate_stamps_and_wide_rows(setting):
    """FFM rows (and 36-float FM rows) keep their stamps in a separate array: load sets every one of them."""
    N, F, D = 400, 15, 10
    for name, d in (("FFM", 4), ("FM", 32)):
        a, oa, c, oc = _resume_case(lambda seed: _model(name, N, F, d, seed), lambda m: _opt(setting, m.parameters()), _eager,
                                    _batches(N, F, 6, seed=8), 3)
        assert c._opt.stamp is not None and c._opt.stamp_col < 0
        assert torch.equal(a._opt.stamp, c._opt.stamp)


GROUPS = [(("LR", "FM", "DeepFM"), 10, 1), (("LR", "FM", "DeepFM"), 32, 4), (("LR", "FM", "DeepFM", "FNN"), 10, 2)]


def _group_batches(N, F, steps, B=256, seed=11):
    g = torch.Generator().manual_seed(seed)
    per = N // F
    out = []
    for _ in range(steps):
        x = (torch.rand(B, F, generator=g) ** 6 * per).long().clamp_(0, per - 1) + torch.arange(F) * per
        out.append((x.to(DEV), (torch.rand(B, generator=g) < 0.3).long().to(DEV)))
    return out


def _make_group(names, N, F, D, max_lines, seed):
    from rl_ctr_prediction_b200 import colocated
    return colocated.colocate([_model(n, N, F, D, seed + i) for i, n in enumerate(names)], max_lines=max_lines)


def _group_step(g, o, x, y):
    return g.train_step(x, y, o).cpu().tolist()


@pytest.mark.parametrize("setting", ["adam_lazy", "adagrad_wd0", "adagrad_wd"])
@pytest.mark.parametrize("names, D, max_lines", GROUPS)
def test_colocated_group_resume(names, D, max_lines, setting):
    N, F = 3000, 15
    _, oa, _, _ = _resume_case(lambda seed: _make_group(names, N, F, D, max_lines, seed),
                               lambda g: _opt(setting, g.parameters()), _group_step, _group_batches(N, F, 6), 3)
    geo = next(e for e in oa.state_dict()["state"].values() if "geometry" in e)["geometry"]
    assert geo["kind"].startswith("group:") and geo["n_rows"] == N


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


def _sharded_step(m, o, x, y):
    return float(m.train_step(x, y, o))


@pytest.mark.parametrize("setting", ["adam_lazy", "adagrad_wd"])
@pytest.mark.parametrize("name", ["LR", "FM", "FFM", "DeepFM", "FNN"])
def test_sharded_world1_resume_and_state_equal_standalone(one_rank, name, setting):
    from rl_ctr_prediction_b200 import pretrain_main, sharded
    N, F, D = 500, 15, 10
    batches = _batches(N, F, 6, seed=2)
    make = lambda seed: sharded.ShardedCTR.from_model(_model(name, N, F, D, seed))
    _, osh, _, _ = _resume_case(make, lambda m: _opt(setting, m.parameters()), _sharded_step, batches, 3)
    single = _model(name, N, F, D, 1)
    o1 = _opt(setting, single.parameters())
    for x, y in batches:
        _eager(single, o1, x, y)
    table = lambda sd: [e for e in sd["state"].values() if "geometry" in e]
    assert_sd_equal(table(o1.state_dict()), table(osh.state_dict()), "table")


@pytest.mark.parametrize("setting", ["adam_lazy", "adagrad_wd"])
def test_sharded_group_world1_resume_and_state_equal_colocated(one_rank, setting):
    from rl_ctr_prediction_b200 import sharded
    names, N, F, D = ("LR", "FM", "DeepFM"), 3001, 15, 10
    batches = _group_batches(N, F, 6, seed=6)
    make = lambda seed: sharded.ShardedGroup.from_group(_make_group(names, N, F, D, 1, seed))
    _, osg, _, _ = _resume_case(make, lambda g: _opt(setting, g.parameters()), _group_step, batches, 3)
    cg = _make_group(names, N, F, D, 1, 1)
    oc = _opt(setting, cg.parameters())
    for x, y in batches:
        _group_step(cg, oc, x, y)
    table = lambda sd: [e for e in sd["state"].values() if "geometry" in e]
    assert_sd_equal(table(oc.state_dict()), table(osg.state_dict()), "joint table")


@pytest.mark.parametrize("setting", ["adam_lazy", "adagrad_wd"])
def test_graphed_resume_and_load_between_replays(setting):
    """Resume into a graphed step; rewind a graphed run by a load between replays (same addresses: the graph is kept); load
    a step past the schedule the graph captured (the graph is captured again) -- each equal to eager steps."""
    from rl_ctr_prediction_b200 import graphs
    names, N, F, D = ("LR", "FM", "DeepFM"), 3000, 15, 10
    batches = _group_batches(N, F, 10, seed=4)
    make = lambda seed, i: _model(names[i], N, F, D, seed + i)
    k = 4
    # eager reference, with its checkpoint at step k
    ref = [make(1, i) for i in range(3)]
    oref = [_opt(setting, m.parameters()) for m in ref]
    lref, ck = [], None
    for s, (x, y) in enumerate(batches):
        if s == k:
            ck = [_save(m, o) for m, o in zip(ref, oref)]
        lref.append([_eager(m, o, x, y) for m, o in zip(ref, oref)])
    # resume into a graphed step
    ms = [make(99, i) for i in range(3)]
    os_ = [_opt(setting, m.parameters()) for m in ms]
    for m, o, c in zip(ms, os_, ck):
        m.load_state_dict(c["model"])
        o.load_state_dict(c["opt"])
    step = graphs.GraphedTrainStep(list(zip(ms, os_)))
    lg = [[float(v) for v in step(x, y)] for x, y in batches[k:]]
    assert step.graph is not None and lg == lref[k:]
    for m, o, r, orr in zip(ms, os_, ref, oref):
        assert_sd_equal((m.state_dict(), o.state_dict()), (r.state_dict(), orr.state_dict()), "graphed resume")
    # a load between replays rewinds to step k: same addresses, the captured graph stays
    g0 = step.graph
    for m, o, c in zip(ms, os_, ck):
        m.load_state_dict(c["model"])
        o.load_state_dict(c["opt"])
    lg = [[float(v) for v in step(x, y)] for x, y in batches[k:]]
    assert step.graph is g0 and lg == lref[k:]
    for m, o, r, orr in zip(ms, os_, ref, oref):
        assert_sd_equal((m.state_dict(), o.state_dict()), (r.state_dict(), orr.state_dict()), "load between replays")
    # a step far past what the captured schedule covers: the next replay must capture again and equal the eager step
    far = copy.deepcopy(ck)
    for c in far:
        for ent in c["opt"]["state"].values():
            ent["step"] = 200000 if isinstance(ent["step"], int) else torch.tensor(200000.0)
    ptrs = [o._captured() for o in os_]
    for m, o, c in zip(ms, os_, far):
        m.load_state_dict(c["model"])
        o.load_state_dict(c["opt"])
    assert [o._captured() for o in os_] != ptrs                # the schedules had to grow
    eg = [make(7, i) for i in range(3)]
    oe = [_opt(setting, m.parameters()) for m in eg]
    for m, o, c in zip(eg, oe, far):
        m.load_state_dict(c["model"])
        o.load_state_dict(c["opt"])
    lg = [[float(v) for v in step(x, y)] for x, y in batches[k:]]
    le = [[_eager(m, o, x, y) for m, o in zip(eg, oe)] for x, y in batches[k:]]
    assert step.graph is not g0 and lg == le
    for m, o, r, orr in zip(ms, os_, eg, oe):
        assert_sd_equal((m.state_dict(), o.state_dict()), (r.state_dict(), orr.state_dict()), "step 200000")
    assert next(e for e in os_[1].state_dict()["state"].values() if "geometry" in e)["step"] == 200000 + len(batches) - k


def test_graphed_callable_captures_again_after_a_load_that_grows_the_schedule():
    from rl_ctr_prediction_b200 import graphs, optim
    torch.manual_seed(0)
    w = torch.nn.Parameter(torch.randn(64, 32, device=DEV))
    w2 = torch.nn.Parameter(w.detach().clone())
    o, o2 = optim.Adam([w], lr=1e-2), optim.Adam([w2], lr=1e-2)

    def fn(p, opt):
        def f(x):
            loss = (p * x).square().sum()
            p.grad = 2 * p * x * x
            opt.step()
            return loss.detach()
        return f
    gc = graphs.GraphedCallable(fn(w, o), [o])
    xs = [torch.randn(64, 32, device=DEV) for _ in range(6)]
    for x in xs[:4]:
        gc(x)
        fn(w2, o2)(x)
    sd = o.state_dict()
    sd["state"][0]["step"] = torch.tensor(200000.0)
    g0 = gc.graph
    o.load_state_dict(sd)
    o2.load_state_dict(sd)
    for x in xs[4:]:
        gc(x)
        fn(w2, o2)(x)
    assert gc.graph is not g0
    torch.cuda.synchronize()
    assert torch.equal(w, w2)
    assert_sd_equal(o.state_dict(), o2.state_dict())


# ---- against stock torch on the CPU port ------------------------------------------------------------------------------------
def _port_pair(name, N, F, D, seed=3):
    from rl_ctr_prediction_b200 import pretrain_main as PM
    torch.manual_seed(seed)
    port = TP.make_port({"W&D": "WideAndDeep", "IPNN": "InnerPNN", "OPNN": "OuterPNN"}.get(name, name), N, F, D)
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


def _port_batches(N, F, steps, B=64, seed=0):
    rng = np.random.default_rng(seed)
    return [(torch.as_tensor(rng.integers(0, N, size=(B, F))), torch.as_tensor((rng.random(B) < 0.3).astype(np.int64)).unsqueeze(1))
            for _ in range(steps)]


def _assert_bar(sd, ref_sd, cls, tower, lr, steps, rtol=2e-5):
    """Every element at 2e-5, with test_gpu_adagrad.py's allowance: a few elements whose gradient nearly cancels -- its last bits
    set by the order of a sum -- may move by up to one step either way.  Adagrad's step does not scale with the gradient; nor
    does Adam's once its moments are that small, and a tower's GEMMs round differently from the CPU's.  Tower-less Adam has no
    allowance (test_gpu_optim.py's bar)."""
    assert set(sd) == set(ref_sd)
    for k, v in ref_sd.items():
        a, b = sd[k].detach().cpu().double().numpy(), v.detach().cpu().double().numpy()
        bad = np.abs(a - b) > rtol * np.abs(b) + rtol * float(np.abs(b).max())
        table = "embedding" in k or k == "linear.weight"
        allowed = max(2e-3 * b.size, 4 if tower else 1) if (table or tower) and (cls == "Adagrad" or tower) else 0
        assert bad.sum() <= allowed, (k, int(bad.sum()), float(np.abs(a - b).max()))
        assert np.abs(a - b).max() <= 2.2 * lr * steps, k


def _port_step(port, popt, x, y):
    return TP.ctr_train_step(port, popt, torch.nn.BCELoss(), x, y)


def _our_step(m, opt, x, y):
    return _eager(m, opt, x.to(DEV), y.to(DEV))


@pytest.mark.parametrize("setting", ["adam_lazy", "adagrad_wd"])
@pytest.mark.parametrize("name", ["FM", "DeepFM", "FFM"])
def test_resume_matches_torch_resume(name, setting):
    from rl_ctr_prediction_b200 import optim
    cls, kw = SETTINGS[setting]
    N, F, D, k, steps = 300, 15, 10, 3, 6
    m, port = _port_pair(name, N, F, D)
    opt, popt = getattr(optim, cls)(m.parameters(), **kw), getattr(torch.optim, cls)(port.parameters(), **kw)
    batches = _port_batches(N, F, steps)
    for x, y in batches[:k]:
        ref, ours = _port_step(port, popt, x, y), _our_step(m, opt, x, y)
        assert abs(ours - ref) <= 1e-5 * max(1.0, abs(ref))
    ck, pck = _save(m, opt), _save(port, popt)
    m2, port2 = _port_pair(name, N, F, D, seed=17)
    m2.load_state_dict(ck["model"])
    port2.load_state_dict(pck["model"])
    opt2, popt2 = getattr(optim, cls)(m2.parameters(), **kw), getattr(torch.optim, cls)(port2.parameters(), **kw)
    opt2.load_state_dict(ck["opt"])
    popt2.load_state_dict(pck["opt"])
    for x, y in batches[k:]:
        ref, ours = _port_step(port2, popt2, x, y), _our_step(m2, opt2, x, y)
        assert abs(ours - ref) <= 1e-5 * max(1.0, abs(ref))
    _assert_bar(m2.state_dict(), port2.state_dict(), cls, name == "DeepFM", kw["lr"], steps)


def _sched(name, opt):
    return {"StepLR": lambda: S.StepLR(opt, 2, 0.5),
            "MultiStepLR": lambda: S.MultiStepLR(opt, [1, 3], 0.3),
            "ExponentialLR": lambda: S.ExponentialLR(opt, 0.8),
            "LambdaLR": lambda: S.LambdaLR(opt, lambda e: 1.0 / (1 + e)),
            "CosineAnnealingLR": lambda: S.CosineAnnealingLR(opt, 4),
            "LinearLR": lambda: S.LinearLR(opt, 0.25, 1.0, 3),
            "SequentialLR": lambda: S.SequentialLR(opt, [S.LinearLR(opt, 0.5, 1.0, 2), S.ExponentialLR(opt, 0.8)], [2]),
            "ReduceLROnPlateau": lambda: S.ReduceLROnPlateau(opt, patience=0, factor=0.5),
            "OneCycleLR": lambda: S.OneCycleLR(opt, max_lr=0.02, total_steps=12, cycle_momentum=False),
            "CyclicLR": lambda: S.CyclicLR(opt, 2e-3, 1e-2, step_size_up=2, cycle_momentum=False)}[name]()


SCHEDS = ["StepLR", "MultiStepLR", "ExponentialLR", "LambdaLR", "CosineAnnealingLR", "LinearLR", "SequentialLR",
          "ReduceLROnPlateau", "OneCycleLR", "CyclicLR"]


@pytest.mark.filterwarnings("ignore::UserWarning")
@pytest.mark.parametrize("cls", ["Adam", "Adagrad"])
@pytest.mark.parametrize("sched", SCHEDS)
def test_schedulers_drive_both_optimizers_and_resume(sched, cls):
    """Five epochs of two steps, the scheduler stepped per epoch (ReduceLROnPlateau on the epoch's loss), optimizer and scheduler
    saved after epoch 2 and restored into new ones on both sides."""
    from rl_ctr_prediction_b200 import optim
    kw = dict(lr=1e-2, weight_decay=1e-5)
    N, F, D, epochs, per = 300, 15, 10, 5, 2
    m, port = _port_pair("FM", N, F, D)
    opt, popt = getattr(optim, cls)(m.parameters(), **kw), getattr(torch.optim, cls)(port.parameters(), **kw)
    sc, psc = _sched(sched, opt), _sched(sched, popt)
    batches = _port_batches(N, F, epochs * per, seed=3)
    lrs = set()
    for e in range(epochs):
        if e == 2:
            ck, pck = _save(m, opt), _save(port, popt)
            ck["sched"], pck["sched"] = sc.state_dict(), psc.state_dict()
            m, port = _port_pair("FM", N, F, D, seed=17)
            m.load_state_dict(ck["model"])
            port.load_state_dict(pck["model"])
            opt, popt = getattr(optim, cls)(m.parameters(), **kw), getattr(torch.optim, cls)(port.parameters(), **kw)
            sc, psc = _sched(sched, opt), _sched(sched, popt)
            opt.load_state_dict(ck["opt"])
            popt.load_state_dict(pck["opt"])
            sc.load_state_dict(ck["sched"])
            psc.load_state_dict(pck["sched"])
        assert opt.param_groups[0]["lr"] == popt.param_groups[0]["lr"], e
        lrs.add(opt.param_groups[0]["lr"])
        tot = 0.0
        for x, y in batches[e * per:(e + 1) * per]:
            ref, ours = _port_step(port, popt, x, y), _our_step(m, opt, x, y)
            assert abs(ours - ref) <= 1e-5 * max(1.0, abs(ref)), (e, ours, ref)
            tot += ref
        if sched == "ReduceLROnPlateau":
            sc.step(1.0)
            psc.step(1.0)
        else:
            sc.step()
            psc.step()
    assert len(lrs) > 1
    _assert_bar(m.state_dict(), port.state_dict(), cls, False, 2e-2, epochs * per)


@pytest.mark.parametrize("cls", ["Adam", "Adagrad"])
def test_dense_only_checkpoints_exchange_with_torch(cls):
    """A tower's parameters: our checkpoint resumes torch.optim, torch's resumes ours, and both continue alike."""
    from rl_ctr_prediction_b200 import optim
    kw = dict(lr=1e-2, weight_decay=1e-4)
    torch.manual_seed(0)
    p0 = [torch.randn(40, 7), torch.randn(33)]
    gs = [[torch.randn_like(p) for p in p0] for _ in range(6)]

    def run(ours_first):
        a = [torch.nn.Parameter(p.clone().to(DEV)) for p in p0]
        b = [torch.nn.Parameter(p.clone().to(DEV)) for p in p0]
        first = getattr(optim if ours_first else torch.optim, cls)(a, **kw)
        for g in gs[:3]:
            for p, gg in zip(a, g):
                p.grad = gg.to(DEV)
            first.step()
        ck = _save(torch.nn.ParameterList(a), first)
        with torch.no_grad():
            for p, q in zip(b, a):
                p.copy_(q)
        second = getattr(torch.optim if ours_first else optim, cls)(b, **kw)
        second.load_state_dict(ck["opt"])
        for g in gs[3:]:
            for p, gg in zip(b, g):
                p.grad = gg.to(DEV)
            second.step()
        return b

    ref = [torch.nn.Parameter(p.clone().to(DEV)) for p in p0]
    ro = getattr(torch.optim, cls)(ref, **kw)
    for g in gs:
        for p, gg in zip(ref, g):
            p.grad = gg.to(DEV)
        ro.step()
    for ours_first in (True, False):
        for p, q in zip(run(ours_first), ref):
            np.testing.assert_allclose(p.detach().cpu().numpy(), q.detach().cpu().numpy(), rtol=2e-5, atol=2e-6)


# ---- a load into an optimizer that has run past the saved step --------------------------------------------------------
@pytest.mark.parametrize("graphed", [False, True])
@pytest.mark.parametrize("setting", ["adam_lazy", "adagrad_wd"])
def test_rewind_after_lr_edits_runs_at_the_checkpoints_lr(setting, graphed):
    """Saved at step k at lr 0.01; the live run then edits lr to 0.001 and back to 0.01 before it is rewound by a load.  The
    steps after the load must all run at 0.01 (the table schedule past step k still held 0.001 for the edited steps)."""
    from rl_ctr_prediction_b200 import graphs
    names, N, F, D, k = ("LR", "FM", "DeepFM"), 3000, 15, 10, 3
    batches = _group_batches(N, F, 10, seed=12)
    make = lambda i: _model(names[i], N, F, D, 1 + i)
    ref = [make(i) for i in range(3)]
    oref = [_opt(setting, m.parameters()) for m in ref]
    lref = [[_eager(m, o, x, y) for m, o in zip(ref, oref)] for x, y in batches]
    ms = [make(i) for i in range(3)]
    os_ = [_opt(setting, m.parameters()) for m in ms]
    step = graphs.GraphedTrainStep(list(zip(ms, os_))) if graphed else \
        (lambda x, y: [_eager(m, o, x, y) for m, o in zip(ms, os_)])
    run = lambda x, y: [float(v) for v in step(x, y)]
    assert [run(x, y) for x, y in batches[:k]] == lref[:k]
    ck = [_save(m, o) for m, o in zip(ms, os_)]
    for s, (x, y) in enumerate(batches[k:]):
        for o in os_:
            o.param_groups[0]["lr"] = 1e-3 if s < 3 else 1e-2
        run(x, y)
    for m, o, c in zip(ms, os_, ck):
        m.load_state_dict(c["model"])
        o.load_state_dict(c["opt"])
        assert o.param_groups[0]["lr"] == 1e-2
    assert [run(x, y) for x, y in batches[k:]] == lref[k:]
    for m, o, r, orr in zip(ms, os_, ref, oref):
        assert_sd_equal((m.state_dict(), o.state_dict()), (r.state_dict(), orr.state_dict()), "rewound")


# ---- refusals on a real table -------------------------------------------------------------------------------------------
def _table_snapshot(m, o):
    t = m._opt
    return (m.table.data.clone(), None if t.stamp is None else t.stamp.clone(), t.step.clone(), t.host_step, t.dirty,
            t.sched.tensor.clone(), t.sched.length, o.lr, o._host_step, tuple(o._dense_count),
            [x.clone() for p in o._dense for x in o._dense_blocks(o._dense_state[p])])


@pytest.mark.parametrize("setting", ["adam_lazy", "adagrad_wd"])
def test_refused_table_loads_leave_the_table_unchanged(setting):
    """Another table geometry (FM D = 10 into FM D = 8 and into LR), a dense state in the table's slot, a table state whose
    tensors have the wrong shape: each refused with its message, the table -- rows, moments or sums, in-record stamps, step
    counters, schedule -- and the dense state bit for bit as they were (rows behind: the refusal must not flush either)."""
    from rl_ctr_prediction_b200 import _lib
    N, F = 400, 15
    src = _model("FM", N, F, 10, 1)
    osrc = _opt(setting, src.parameters())
    for x, y in _batches(N, F, 3, seed=3):
        _eager(src, osrc, x, y)
    sd = osrc.state_dict()
    ti = next(i for i, e in sd["state"].items() if "geometry" in e)
    di = next(i for i, e in sd["state"].items() if "geometry" not in e)
    for name, d in (("FM", 8), ("LR", 1)):
        m = _model(name, N, F, d, 2)
        o = _opt(setting, m.parameters())
        bs = _batches(N, F, 5, seed=4)
        for x, y in bs[:4]:
            _eager(m, o, x, y)
        mine = o.state_dict()                                # (flushes)
        _eager(m, o, *bs[4])
        assert m._opt.dirty == m._opt.lazy                   # lazy tables have rows behind again: a flush would show
        before = _table_snapshot(m, o)
        mt = next(i for i, e in mine["state"].items() if "geometry" in e)
        bad_geo = copy.deepcopy(mine)
        bad_geo["state"][mt] = sd["state"][ti]
        dense_in_table = copy.deepcopy(mine)
        dense_in_table["state"][mt] = copy.deepcopy(sd["state"][di])
        bad_shape = copy.deepcopy(mine)
        for k in m._opt._blocks():
            bad_shape["state"][mt][k] = bad_shape["state"][mt][k][:-1]
        for bad, msg in ((bad_geo, r"\['geometry'\] is .* but this table's is"),
                         (dense_in_table, "is a dense parameter's state, but parameter .* is an embedding table"),
                         (bad_shape, "has the shape")):
            with pytest.raises(_lib.RlctrError, match=msg):
                o.load_state_dict(bad)
            after = _table_snapshot(m, o)
            for u, v in zip(before, after):
                if isinstance(u, list):
                    assert all(torch.equal(a, b) for a, b in zip(u, v))
                else:
                    assert torch.equal(u, v) if isinstance(u, torch.Tensor) else u == v
