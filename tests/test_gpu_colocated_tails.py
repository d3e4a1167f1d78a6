"""Co-located groups with the tower-tail models (rl_ctr_prediction_b200/colocated.py): FNN, InnerPNN, OuterPNN, DCN and AFM share
the joint record with LR / FM / DeepFM / WideAndDeep.  Every vector member must give the numbers of its stand-alone model bit for
bit -- losses, every row of its table, every dense parameter, the dropout counters -- and LR agrees to rounding, as in
tests/test_gpu_colocated.py.  The tail member appears both first and last in the combinations below.
"""
import copy

import numpy as np
import pytest
import torch

from conftest import state_from_golden

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
F, D = 15, 10
# class name -> get_model name
NAMES = {"LR": "LR", "FM": "FM", "DeepFM": "DeepFM", "WideAndDeep": "W&D", "FNN": "FNN", "InnerPNN": "IPNN", "OuterPNN": "OPNN",
         "DCN": "DCN", "AFM": "AFM", "FFM": "FFM"}
TAILS = ("FNN", "InnerPNN", "OuterPNN", "DCN", "AFM")
COMBOS = [("LR", "FM", "FNN"), ("InnerPNN", "DeepFM"), ("DCN", "WideAndDeep"), ("FM", "AFM"), ("OuterPNN", "LR", "FM"),
          ("AFM", "LR", "DCN")]


def _towers(m):
    from rl_ctr_prediction_b200 import mlp
    return [t for t in m.modules() if isinstance(t, mlp.Tower)]


def _set_dropout(m, on, seed):
    """Dropout of the towers (train / eval) and AFM's always-on attention dropout (0.2 / 0), with the counter-hash states set
    explicitly: a deep copy then starts from the same masks."""
    for k, t in enumerate(_towers(m)):
        t.train(on)
        t._rlctr_rng = torch.tensor([seed + 17 * k, 0], dtype=torch.int64, device=DEV)
    if type(m).__name__ == "AFM":
        m.dropout_p = 0.2 if on else 0.0
        m._rlctr_rng = torch.tensor([seed + 101, 0], dtype=torch.int64, device=DEV)


def _rng_counters(m):
    out = [int(t._rlctr_rng[1]) for t in _towers(m)]
    if type(m).__name__ == "AFM":
        out.append(int(m._rlctr_rng[1]))
    return out


@pytest.fixture
def make_models():
    from rl_ctr_prediction_b200 import pretrain_main as PM

    def make(names, N, seed=3, dropout=False):
        torch.manual_seed(seed)
        ms = [PM.get_model(NAMES[n], N, F, D).to(DEV).train() for n in names]
        for i, m in enumerate(ms):
            _set_dropout(m, dropout, 1000 * seed + 10 * i)
        return ms
    return make


@pytest.fixture
def make_batches():
    def make(N, B, steps, seed=11, zipf=False):
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
    return make


def _train_separate(models, batches, mode="lazy"):
    from rl_ctr_prediction_b200 import graphs, optim
    opts = [optim.Adam(m.parameters(), lr=1e-3, weight_decay=1e-5, mode=mode) for m in models]
    loss_fn = torch.nn.BCELoss()
    return np.array([[float(graphs.eager_step(m, o, loss_fn, x, y)) for m, o in zip(models, opts)] for x, y in batches])


def _train_group(models, batches, mode="lazy"):
    from rl_ctr_prediction_b200 import colocated, optim
    group = colocated.colocate(models)
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


@pytest.mark.parametrize("mode", ["lazy", "dense"])
@pytest.mark.parametrize("zipf", [False, True])
@pytest.mark.parametrize("names", COMBOS)
def test_tail_group_equals_standalone(make_models, make_batches, names, zipf, mode):
    N, B, steps = 3000, 512, 5
    sep = make_models(names, N)
    grp = [copy.deepcopy(m) for m in sep]
    batches = make_batches(N, B, steps, zipf=zipf)
    l_sep = _train_separate(sep, batches, mode)
    group, l_grp = _train_group(grp, batches, mode)
    assert group._geom.row_stride <= 32
    _assert_same(names, sep, grp, l_sep, l_grp)


@pytest.mark.parametrize("names", COMBOS)
def test_tail_group_dropout_on(make_models, make_batches, names):
    """Towers in train(), AFM's attention dropout at 0.2: the group step draws and advances each member's own counter exactly as
    the stand-alone step does."""
    N, B, steps = 2500, 384, 4
    sep = make_models(names, N, seed=7, dropout=True)
    grp = [copy.deepcopy(m) for m in sep]
    batches = make_batches(N, B, steps, seed=5)
    l_sep = _train_separate(sep, batches)
    _, l_grp = _train_group(grp, batches)
    _assert_same(names, sep, grp, l_sep, l_grp)
    for a, b, n in zip(sep, grp, names):
        ca, cb = _rng_counters(a), _rng_counters(b)
        assert ca == cb, n
        if n in TAILS or n in ("DeepFM", "WideAndDeep"):
            assert ca and all(c > 0 for c in ca), n                      # the masks were drawn


@pytest.mark.parametrize("mode", ["lazy", "dense"])
@pytest.mark.parametrize("pos", ["first", "last"])
@pytest.mark.parametrize("tail", TAILS)
def test_tail_member_matches_reference_trajectory(golden, golden_tails, tail, pos, mode):
    """Three steps of the reference loop body (tests/golden/make_golden_tails.py: the real p_model classes, dense torch.optim.Adam)
    for a tail member trained inside a group with FM and LR: pCTR, loss and final parameters, with the tolerances of
    test_gpu_models.py::test_tail_models_match_reference (AFM's dropout off there and here)."""
    from test_gpu_models import assert_state, build, close, load
    from rl_ctr_prediction_b200 import colocated, optim
    names = (tail, "FM", "LR") if pos == "first" else ("LR", "FM", tail)
    src = {n: (golden_tails if n == tail else golden) for n in names}
    members = []
    for n in names:
        m = load(build(NAMES[n], 255), state_from_golden(src[n], f"train/{n}/init")).to(DEV)
        if n == "AFM":
            m.dropout_p = 0.0
        members.append(m.eval())
    group = colocated.colocate(members)
    opt = optim.Adam(group.parameters(), lr=1e-3, weight_decay=1e-5, mode=mode)
    xs, ys = golden["train/x"], golden["train/y"]
    for s in range(3):
        x, y = torch.as_tensor(xs[s]).to(DEV), torch.as_tensor(ys[s]).to(DEV)
        p = group(x)
        losses = group.train_step(x, y, opt)
        for i, n in enumerate(names):
            close(p[:, i:i + 1], src[n][f"train/{n}/pctr{s}"])
            close(losses[i], src[n][f"train/{n}/loss{s}"])
    for m, n in zip(members, names):
        assert_state(m, state_from_golden(src[n], f"train/{n}/final"))


@pytest.mark.parametrize("names", COMBOS)
def test_tail_group_inference_and_checkpoints(golden_tails, make_models, make_batches, names):
    from rl_ctr_prediction_b200 import pretrain_main as PM
    N, B = 2000, 300
    sep = make_models(names, N, seed=13)
    members = [copy.deepcopy(m) for m in sep]
    batches = make_batches(N, B, 3, seed=3)
    _train_separate(sep, batches)
    group, _ = _train_group(members, batches)
    x = batches[0][0]
    with torch.no_grad():
        for m in sep + members:
            m.eval()
        want = torch.cat([m(x) for m in sep], dim=1)
        got = group(x)                                    # one gather, [B, M]
        per_member = torch.cat([m(x) for m in members], dim=1)
    assert got.shape == (B, len(names))
    for i, n in enumerate(names):
        if n == "LR":
            torch.testing.assert_close(got[:, i], want[:, i], rtol=1e-6, atol=1e-7)
        else:
            assert torch.equal(got[:, i], want[:, i]), n       # the group kernel and the tail reproduce the stand-alone model
        if n in ("FNN", "InnerPNN", "OuterPNN", "DCN"):
            assert torch.equal(per_member[:, i], got[:, i]), n  # no table part: the member's own gather copies the same rows
        else:
            # a member called on its own sums its table part over the wider joint row in another order (rounding level)
            torch.testing.assert_close(per_member[:, i], got[:, i], rtol=1e-4, atol=1e-5)
    # reference keys and shapes; load_state_dict round-trips through the joint record
    torch.manual_seed(99)
    for i, n in enumerate(names):
        sd = members[i].state_dict()
        if n in TAILS:
            assert set(sd) == set(state_from_golden(golden_tails, f"train/{n}/init")), n
        ref_sd = sep[i].state_dict()
        assert {k: tuple(v.shape) for k, v in sd.items()} == {k: tuple(v.shape) for k, v in ref_sd.items()}, n
        fresh = PM.get_model(NAMES[n], N, F, D).to(DEV).eval()
        if n == "AFM":
            fresh.dropout_p = 0.0
        new_sd = {k: v.clone() for k, v in fresh.state_dict().items()}
        members[i].load_state_dict(new_sd)
        for k, v in members[i].state_dict().items():
            assert torch.equal(v, new_sd[k]), (n, k)
        with torch.no_grad():
            a, b = group(x)[:, i], fresh(x)[:, 0]
        if n == "LR":
            torch.testing.assert_close(a, b, rtol=1e-6, atol=1e-7)
        else:
            assert torch.equal(a, b), n
    for i, n in enumerate(names):
        if n == "FNN":                                    # an FM checkpoint's embedding, through the joint record
            fm = PM.get_model("FM", N, F, D).state_dict()
            members[i].load_embedding(fm)
            assert torch.equal(members[i].state_dict()["feature_embedding.weight"].cpu(), fm["feature_embedding.weight"])


@pytest.mark.parametrize("names", [("LR", "FM", "FNN"), ("AFM", "LR", "DCN"), ("InnerPNN", "OuterPNN")])
def test_tail_group_lazy_flush_equals_dense(make_models, make_batches, names):
    """lazy + flush == dense Adam on a joint record with tail members, with rows that stay untouched for many steps."""
    N, B, steps = 6000, 64, 30
    a = make_models(names, N, seed=5)
    b = [copy.deepcopy(m) for m in a]
    batches = make_batches(N, B, steps, seed=2)
    ga, la = _train_group(a, batches, mode="lazy")
    gb, lb = _train_group(b, batches, mode="dense")
    assert np.array_equal(la, lb)
    ga.flush()
    gb.flush()
    assert torch.equal(ga.table.data, gb.table.data)
    for ma, mb in zip(a, b):
        for (k, u), (_, v) in zip(ma.state_dict().items(), mb.state_dict().items()):
            assert torch.equal(u, v), k


@pytest.mark.parametrize("names", [("LR", "FM", "FNN"), ("DCN", "AFM"), ("LR", "InnerPNN", "OuterPNN")])
def test_tail_group_graphed_step_equals_eager(make_models, make_batches, names):
    """GraphedTrainStep of a group with tail members, dropout on (the device counters are replayed too) == the eager steps."""
    from rl_ctr_prediction_b200 import colocated, graphs, optim
    N, B, steps = 4000, 256, 7
    a = make_models(names, N, seed=9, dropout=True)
    b = [copy.deepcopy(m) for m in a]
    batches = make_batches(N, B, steps, seed=4)
    ga, gb = colocated.colocate(a), colocated.colocate(b)
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
    for ma, mb in zip(a, b):
        assert _rng_counters(ma) == _rng_counters(mb)


@pytest.mark.parametrize("B", [1, 7, 257])
@pytest.mark.parametrize("names", [("FNN", "LR", "FM"), ("WideAndDeep", "DCN"), ("LR", "InnerPNN", "AFM")])
def test_tail_group_ragged_batches_and_out_of_range_ids(make_models, names, B):
    """Odd batch sizes and ids outside the vocabulary (zero row, no update): the group follows the stand-alone models."""
    N, steps = 500, 3
    sep = make_models(names, N, seed=41)
    grp = [copy.deepcopy(m) for m in sep]
    g = torch.Generator().manual_seed(3)
    batches = []
    for _ in range(steps):
        x = torch.randint(0, N, (B, F), generator=g)
        x[0, 0] = N + 7
        x[-1, 3] = -1
        batches.append((x.to(DEV), (torch.rand(B, generator=g) < 0.5).long().to(DEV)))
    l_sep = _train_separate(sep, batches)
    _, l_grp = _train_group(grp, batches)
    _assert_same(names, sep, grp, l_sep, l_grp)


@pytest.mark.parametrize("names", [("FM", "FNN", "DeepFM"), ("AFM", "DCN", "InnerPNN"), ("LR", "OuterPNN", "FNN", "WideAndDeep"),
                                   ("FM", "FFM"), ("FFM", "DCN")])
def test_tail_groups_that_do_not_fit(make_models, names):
    from rl_ctr_prediction_b200 import _lib, colocated
    ms = make_models(names, 300)
    with pytest.raises(_lib.RlctrError, match="FFM|32 floats"):
        colocated.colocate(ms)


def test_tail_member_joins_once(make_models):
    from rl_ctr_prediction_b200 import _lib, colocated
    fm, fnn, dcn = make_models(("FM", "FNN", "DCN"), 300)
    colocated.colocate([fm, fnn])
    with pytest.raises(_lib.RlctrError, match="once"):
        colocated.colocate([fnn, dcn])
