"""optim.Adam / optim.Adagrad as torch.optim.Optimizers, without a GPU: torch's LR schedulers drive them, a second parameter
group is refused, state_dict() has torch's structure and keys, and every refusal of load_state_dict leaves the optimizer as it
was (dense parameters on the CPU: construction, state_dict and load_state_dict launch nothing)."""
import copy

import pytest
import torch
from torch.optim import lr_scheduler as S

from rl_ctr_prediction_b200 import _lib, optim


def _params(seed=0):
    g = torch.Generator().manual_seed(seed)
    return [torch.nn.Parameter(torch.randn(5, 3, generator=g)), torch.nn.Parameter(torch.randn(4, generator=g))]


def _schedulers(opt):
    return {
        "StepLR": lambda: S.StepLR(opt, 2, 0.5),
        "MultiStepLR": lambda: S.MultiStepLR(opt, [1, 3], 0.3),
        "ExponentialLR": lambda: S.ExponentialLR(opt, 0.9),
        "LambdaLR": lambda: S.LambdaLR(opt, lambda e: 1.0 / (1 + e)),
        "CosineAnnealingLR": lambda: S.CosineAnnealingLR(opt, 4),
        "LinearLR": lambda: S.LinearLR(opt, 0.25, 1.0, 3),
        "SequentialLR": lambda: S.SequentialLR(opt, [S.LinearLR(opt, 0.5, 1.0, 2), S.ExponentialLR(opt, 0.8)], [2]),
        "ReduceLROnPlateau": lambda: S.ReduceLROnPlateau(opt, patience=0, factor=0.5),
        "OneCycleLR": lambda: S.OneCycleLR(opt, max_lr=0.05, total_steps=10, cycle_momentum=False),
        "CyclicLR": lambda: S.CyclicLR(opt, 1e-3, 1e-2, step_size_up=2, cycle_momentum=False),
    }


KW = {"Adam": dict(lr=1e-2, weight_decay=1e-5), "Adagrad": dict(lr=1e-2, weight_decay=1e-4)}
OPTS = {"Adam": lambda ps: optim.Adam(ps, **KW["Adam"]), "Adagrad": lambda ps: optim.Adagrad(ps, **KW["Adagrad"])}
TORCH = {"Adam": torch.optim.Adam, "Adagrad": torch.optim.Adagrad}


@pytest.mark.parametrize("cls", list(OPTS))
def test_is_a_torch_optimizer(cls):
    assert isinstance(OPTS[cls](_params()), torch.optim.Optimizer)


@pytest.mark.filterwarnings("ignore:Detected call of `lr_scheduler.step()` before `optimizer.step()`")
@pytest.mark.parametrize("sched", list(_schedulers(None)))
@pytest.mark.parametrize("cls", list(OPTS))
def test_schedulers_edit_lr(cls, sched):
    """Each scheduler builds on our optimizer and moves lr exactly as it moves torch's; _sync_hyper accepts every value."""
    ours, ref = OPTS[cls](_params()), TORCH[cls](_params(), lr=1e-2)
    s_ours, s_ref = _schedulers(ours)[sched](), _schedulers(ref)[sched]()
    seen = set()
    for e in range(6):
        assert ours.param_groups[0]["lr"] == ref.param_groups[0]["lr"], e
        seen.add(ours.param_groups[0]["lr"])
        ours._sync_hyper()
        assert ours.lr == ours.param_groups[0]["lr"]
        if sched == "ReduceLROnPlateau":
            s_ours.step(1.0)
            s_ref.step(1.0)
        else:
            s_ours.step()
            s_ref.step()
    assert len(seen) > 1


def test_one_cycle_with_momentum_edits_betas_and_the_step_refuses():
    ours = OPTS["Adam"](_params())
    S.OneCycleLR(ours, max_lr=0.05, total_steps=10, cycle_momentum=True)
    assert ours.param_groups[0]["betas"] != (0.9, 0.999)
    with pytest.raises(_lib.RlctrError, match="changing betas after construction"):
        ours._sync_hyper()


@pytest.mark.parametrize("cls", list(OPTS))
def test_torch_keys_are_fixed(cls):
    o = OPTS[cls](_params())
    assert sorted(o.param_groups[0]) == sorted(TORCH[cls](_params()).param_groups[0])
    for k, v in o._TORCH_KEYS.items():
        assert o.param_groups[0][k] == v
        o.param_groups[0][k] = True if v is not True else False
        with pytest.raises(_lib.RlctrError, match=f"changing {k} after construction"):
            o._sync_hyper()
        o.param_groups[0][k] = v
    o._sync_hyper()


@pytest.mark.parametrize("cls", list(OPTS))
def test_one_parameter_group(cls):
    ps = _params()
    with pytest.raises(_lib.RlctrError, match="one parameter group"):
        type(OPTS[cls](ps))([{"params": ps[:1]}, {"params": ps[1:]}])
    o = OPTS[cls](ps[:1])
    with pytest.raises(_lib.RlctrError, match="one parameter group"):
        o.add_param_group({"params": ps[1:]})
    assert len(o.param_groups) == 1 and len(o.param_groups[0]["params"]) == 1


@pytest.mark.parametrize("cls", list(OPTS))
def test_never_stepped_state_dict_has_torch_keys(cls):
    ps = _params()
    ours, ref = OPTS[cls](ps), TORCH[cls](ps, **KW[cls])
    a, b = ours.state_dict(), ref.state_dict()
    assert set(a) == {"state", "param_groups"}
    assert sorted(a["param_groups"][0]) == sorted(b["param_groups"][0])
    assert a["param_groups"][0]["params"] == b["param_groups"][0]["params"] == [0, 1]
    assert sorted(a["state"]) == sorted(b["state"])             # Adam: none yet; Adagrad: every parameter from construction on
    for i, ent in b["state"].items():
        assert sorted(a["state"][i]) == sorted(ent)
        for k, v in ent.items():
            assert a["state"][i][k].dtype == v.dtype and a["state"][i][k].shape == v.shape and torch.equal(a["state"][i][k], v)
    ours.load_state_dict(b)                                     # and torch's loads into ours
    ref.load_state_dict(a)                                      # and ours into torch's


def _stepped(cls):
    """An optimizer whose dense state was loaded from torch's after three steps (no kernel runs on the CPU)."""
    ps = _params()
    ref = TORCH[cls](ps, **KW[cls])
    for _ in range(3):
        for p in ps:
            p.grad = torch.ones_like(p)
        ref.step()
    o = OPTS[cls](_params(1))
    o.load_state_dict(ref.state_dict())
    return o, ref.state_dict()


def _snapshot(o):
    return copy.deepcopy((o.param_groups[0] | {"params": None}, o._dense_count, o._host_step, o.lr,
                          {o._dense_index[p]: [t.clone() for t in o._dense_blocks(st)] for p, st in o._dense_state.items()},
                          None if o._dense_steps is None else o._dense_steps.clone(),
                          None if o._dense_sched is None else o._dense_sched.tensor.clone()))


def _assert_same(a, b):
    assert a[:4] == b[:4]
    assert a[4].keys() == b[4].keys()
    for k in a[4]:
        assert all(torch.equal(x, y) for x, y in zip(a[4][k], b[4][k]))
    for x, y in zip(a[5:], b[5:]):
        assert (x is None and y is None) or torch.equal(x, y)


def _refusals(cls, good):
    other = "Adagrad" if cls == "Adam" else "Adam"
    o_other, sd_other = _stepped(other)
    fixed = OPTS[cls](_params())._FIXED[-1]

    def edit(fn):
        sd = copy.deepcopy(good)
        fn(sd)
        return sd

    def fix(sd):
        k = fixed
        sd["param_groups"][0][k] = sd["param_groups"][0][k] * 2 + 1e-3

    return [
        (sd_other, _lib.RlctrError, "not .*'s state"),
        (o_other.state_dict(), _lib.RlctrError, "not .*'s state"),
        (edit(lambda sd: sd["param_groups"][0]["params"].pop()), ValueError, "doesn't match the size"),
        (edit(lambda sd: sd["param_groups"].append(dict(sd["param_groups"][0]))), ValueError, "number of parameter groups"),
        (edit(lambda sd: sd["state"][1].update({k: torch.zeros(5) for k in sd["state"][1] if k != "step"})),
         _lib.RlctrError, r"state\[1\]\['(exp_avg|sum)'\] has the shape"),
        (edit(fix), _lib.RlctrError, f"construct the optimizer with {fixed}="),
        (edit(lambda sd: sd["param_groups"][0].update(maximize=True)), _lib.RlctrError, "only maximize=False"),
        (edit(lambda sd: sd["state"][0].update(geometry={"n_rows": 5})), _lib.RlctrError, r"state\[0\] is an embedding table's"),
        (edit(lambda sd: sd["state"][0].update(step=torch.tensor(-1.0))), _lib.RlctrError, r"state\[0\]\['step'\]"),
    ]


@pytest.mark.parametrize("cls", list(OPTS))
def test_refused_loads_change_nothing(cls):
    o, good = _stepped(cls)
    before = _snapshot(o)
    for sd, exc, msg in _refusals(cls, good):
        with pytest.raises(exc, match=msg):
            o.load_state_dict(sd)
        _assert_same(_snapshot(o), before)
    o.load_state_dict(good)
    _assert_same(_snapshot(o), before)


@pytest.mark.parametrize("cls", list(OPTS))
def test_lr_and_extra_keys_come_from_the_checkpoint(cls):
    o, good = _stepped(cls)
    sd = copy.deepcopy(good)
    sd["param_groups"][0]["lr"] = 0.123
    sd["param_groups"][0]["initial_lr"] = 0.5
    o.load_state_dict(sd)
    assert o.lr == 0.123 and o.param_groups[0]["initial_lr"] == 0.5 and o._dense_count == [3, 3]
    assert o.state_dict()["param_groups"] == sd["param_groups"]
    o._sync_hyper()


@pytest.mark.parametrize("cls", list(OPTS))
def test_dense_state_round_trips_with_torch(cls):
    o, good = _stepped(cls)
    sd = o.state_dict()
    for i, ent in good["state"].items():
        assert sorted(sd["state"][i]) == sorted(ent)
        for k, v in ent.items():
            assert sd["state"][i][k].dtype == v.dtype and sd["state"][i][k].shape == v.shape, (i, k)
            assert torch.equal(sd["state"][i][k], v), (i, k)
        assert sd["state"][i]["step"].device.type == "cpu" and sd["state"][i]["step"].dim() == 0
    ref = TORCH[cls](_params(2), **dict(KW[cls], lr=1.0))
    ref.load_state_dict(sd)
    assert ref.param_groups[0]["lr"] == 1e-2
    ps = _params()
    for p in ps:
        p.grad = torch.ones_like(p)
    ref.step()                                                  # torch steps from our state
    fresh = OPTS[cls](_params())
    fresh.load_state_dict({"state": {}, "param_groups": sd["param_groups"]})    # no entries: every parameter afresh
    assert fresh._dense_count == [0, 0]


@pytest.mark.parametrize("kind", ["Adam", "Adagrad"])
def test_forced_retabulation_after_a_rewind(kind):
    """A load moves the step back: the entries after the saved step may hold lrs edited after it, and the checkpoint's lr may
    equal the live one.  set_lr(..., force=True), which load_state_dict uses, rewrites them all the same."""
    from rl_ctr_prediction_b200.tables import AdagradSchedule, AdamSchedule
    make = (lambda lr: AdamSchedule(lr, (0.9, 0.999), "cpu", length=64)) if kind == "Adam" else \
        (lambda lr: AdagradSchedule(lr, 0.05, "cpu", length=64))
    s = make(0.01)
    s.set_lr(0.001, 6)                  # edited after step 5 ...
    s.set_lr(0.01, 11)                  # ... and back after step 10
    s.ensure(5)
    s.set_lr(0.01, 4)                   # an unchanged lr returns at once: steps 6..10 keep 0.001
    assert not torch.equal(s.tensor[4:], make(0.01).tensor[4:])
    s.set_lr(0.01, 4, force=True)       # a load resuming after step 3 at lr 0.01
    assert torch.equal(s.tensor[4:], make(0.01).tensor[4:])
