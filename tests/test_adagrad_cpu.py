"""optim.Adagrad without a GPU: the Adagrad entry points refuse bad arguments and unsupported shapes before any CUDA call, the
clr table is torch.optim.Adagrad's own per-step scalar, and the constructor validates its arguments like torch's."""
import ctypes as C

import pytest
import torch

from rl_ctr_prediction_b200 import _lib

EINVAL, EUNSUPPORTED, EWORKSPACE = -1, -2, -3
_FAKE = 1 << 20                     # 16-byte aligned stand-in address: every call below returns before reading through it


def _ada(stamp_col=-1, stamp=None, state=_FAKE, clr=_FAKE):
    return _lib.Adagrad(state, stamp, clr, _FAKE, 8192, stamp_col, 1e-10, 1e-5)


def test_rows_adagrad_refuses_before_touching_memory():
    lib = _lib.load()
    g = _lib.RowGrad(None, _FAKE, _FAKE, None, 15, 0)
    fm = _lib.Table(_FAKE, 1000, 16, 0, 1, 10, 48)
    ws_need = lib.rlctr_rows_ws_bytes(64)
    call = lambda t, a, n=64, ws=_FAKE, wsb=ws_need: lib.rlctr_rows_adagrad(_FAKE, _FAKE, n, C.byref(g), C.byref(t), C.byref(a), ws,
                                                                           wsb, None)
    assert call(fm, _ada(), n=-1) == EINVAL
    assert call(fm, _ada(state=None)) == EINVAL
    assert call(fm, _ada(clr=None)) == EINVAL
    assert call(fm, _ada(stamp_col=48)) == EINVAL                                    # stamp past the record
    assert call(fm, _ada(), wsb=ws_need - 1) == EWORKSPACE
    assert call(fm, _ada(), ws=None) == EWORKSPACE
    ffm = _lib.Table(_FAKE, 1000, 516, 15 * 34, 0, 15 * 34, 3 * 516)                 # FFM, F = 15, D = 34: 516 floats
    assert call(ffm, _ada()) == EUNSUPPORTED
    wide = _lib.Table(_FAKE, 1000, 36, 0, 1, 32, 108)
    assert call(wide, _ada(stamp_col=35)) == EUNSUPPORTED                            # wide rows keep separate stamps
    with pytest.raises(_lib.RlctrError, match=r"at most 512 floats"):
        _lib.call("rlctr_rows_adagrad", lib.rlctr_rows_adagrad, _FAKE, _FAKE, 64, C.byref(g), C.byref(ffm), C.byref(_ada()), _FAKE,
                  ws_need, None, key="rlctr_rows_adagrad[FFM]")


def test_group_rows_adagrad_refuses_before_touching_memory():
    lib = _lib.load()
    members = (_lib.Member * 2)()
    members[0].lin_col, members[0].emb_col, members[0].dim, members[0].dlogit = 0, 0, 0, _FAKE
    members[1].lin_col, members[1].emb_col, members[1].dim, members[1].flags, members[1].dlogit = 1, 2, 10, 1, _FAKE
    t = _lib.Table(_FAKE, 1000, 16, -1, 0, 12, 96)
    ws_need = lib.rlctr_rows_ws_bytes(64)
    call = lambda t, a, m=2, ws=ws_need, fields=15: lib.rlctr_group_rows_adagrad(_FAKE, _FAKE, 64, C.byref(t), C.byref(a), members, m,
                                                                                _FAKE, 0, fields, 1, None, _FAKE, ws, None)
    assert call(t, _ada(stamp_col=12), m=0) == EINVAL
    assert call(t, _ada(stamp_col=12), m=5) == EINVAL
    assert call(t, _ada(stamp_col=12), fields=0) == EINVAL
    assert call(t, _ada(state=None)) == EINVAL
    assert call(t, _ada(stamp_col=5)) == EINVAL                                      # the stamp on a member column
    assert call(t, _ada(stamp_col=12), ws=16) == EWORKSPACE
    big = _lib.Table(_FAKE, 1000, 132, -1, 0, 130, 396)
    assert call(big, _ada()) == EUNSUPPORTED                                         # past four lines
    with pytest.raises(_lib.RlctrError, match=r"at most 128 floats"):
        _lib.call("rlctr_group_rows_adagrad", lib.rlctr_group_rows_adagrad, _FAKE, _FAKE, 64, C.byref(big), C.byref(_ada()), members,
                  2, _FAKE, 0, 15, 1, None, _FAKE, ws_need, None)


def test_catchup_and_flush_refuse_before_touching_memory():
    lib = _lib.load()
    t = _lib.Table(_FAKE, 1000, 16, 0, 1, 10, 48)
    assert lib.rlctr_adagrad_catchup(_FAKE, 64, C.byref(t), C.byref(_ada()), None) == EINVAL            # no stamps: nothing to replay
    assert lib.rlctr_adagrad_flush(C.byref(t), C.byref(_ada()), 0, 1000, None) == EINVAL
    assert lib.rlctr_adagrad_catchup(_FAKE, -1, C.byref(t), C.byref(_ada(stamp_col=11)), None) == EINVAL
    assert lib.rlctr_adagrad_catchup(None, 64, C.byref(t), C.byref(_ada(stamp_col=11)), None) == EINVAL
    assert lib.rlctr_adagrad_flush(C.byref(t), C.byref(_ada(stamp_col=11)), 0, 1001, None) == EINVAL    # past the table
    assert lib.rlctr_adagrad_flush(C.byref(t), C.byref(_ada(stamp_col=11, clr=None)), 0, 1000, None) == EINVAL
    assert lib.rlctr_adagrad_flush(C.byref(t), C.byref(_ada(stamp_col=11)), 5, 5, None) == 0             # empty range: no launch
    odd = _lib.Table(_FAKE, 1000, 6, 0, 1, 4, 18)
    assert lib.rlctr_adagrad_catchup(_FAKE, 64, C.byref(odd), C.byref(_ada(stamp_col=5)), None) == EUNSUPPORTED
    big = _lib.Table(_FAKE, 1000, 132, -1, 0, 129, 396)                              # 33 chunks with an in-record stamp
    assert lib.rlctr_adagrad_flush(C.byref(big), C.byref(_ada(stamp_col=129)), 0, 1000, None) == EUNSUPPORTED
    assert lib.rlctr_adagrad_catchup(_FAKE, 64, C.byref(big), C.byref(_ada(stamp_col=129)), None) == EUNSUPPORTED
    with pytest.raises(_lib.RlctrError, match=r"at most 128 floats"):
        _lib.call("rlctr_adagrad_flush", lib.rlctr_adagrad_flush, C.byref(big), C.byref(_ada(stamp_col=129)), 0, 1000, None)


def test_dense_adagrad_multi_refuses_before_touching_memory():
    lib = _lib.load()
    k = 25
    ptrs = (C.c_void_p * k)(*([_FAKE] * k))
    sizes = (C.c_int64 * k)(*([10] * k))
    idx = (C.c_int32 * k)(*range(k))
    assert lib.rlctr_dense_adagrad_multi(ptrs, ptrs, ptrs, sizes, k, _FAKE, _FAKE, idx, 1e-10, 0.0, None) == EUNSUPPORTED
    assert lib.rlctr_dense_adagrad_multi(ptrs, ptrs, ptrs, sizes, 2, None, _FAKE, idx, 1e-10, 0.0, None) == EINVAL
    assert lib.rlctr_dense_adagrad_multi(ptrs, ptrs, None, sizes, 2, _FAKE, _FAKE, idx, 1e-10, 0.0, None) == EINVAL
    assert lib.rlctr_dense_adagrad_multi(ptrs, ptrs, ptrs, sizes, -1, _FAKE, _FAKE, idx, 1e-10, 0.0, None) == EINVAL
    assert lib.rlctr_dense_adagrad_multi(ptrs, ptrs, ptrs, sizes, 0, _FAKE, _FAKE, idx, 1e-10, 0.0, None) == 0
    bad = (C.c_int64 * 2)(10, -1)
    assert lib.rlctr_dense_adagrad_multi(ptrs, ptrs, ptrs, bad, 2, _FAKE, _FAKE, idx, 1e-10, 0.0, None) == EINVAL
    neg = (C.c_int32 * 2)(0, -1)
    assert lib.rlctr_dense_adagrad_multi(ptrs, ptrs, ptrs, sizes, 2, _FAKE, _FAKE, neg, 1e-10, 0.0, None) == EINVAL


def _torch_clr(lr, lr_decay, steps, edit=None):
    """The clr torch.optim.Adagrad applies at each step, read off the optimizer itself: with grad 1, state_sum 0 and eps 0
    the step is p = 0 + (-clr) * 1 / (sqrt(1) + 0) = -float32(clr) exactly; p and the sum are reset after each step."""
    p = torch.nn.Parameter(torch.zeros(1))
    opt = torch.optim.Adagrad([p], lr=lr, lr_decay=lr_decay, eps=0.0)
    out = [0.0]
    for t in range(1, steps + 1):
        if edit is not None and t == edit[0]:
            opt.param_groups[0]["lr"] = edit[1]
        p.grad = torch.ones(1)
        with torch.no_grad():
            p.zero_()
            opt.state[p]["sum"].zero_()
        opt.step()
        out.append(-float(p.item()))
    return torch.tensor(out, dtype=torch.float32)


@pytest.mark.parametrize("lr, lr_decay", [(1e-2, 0.0), (0.05, 1e-3), (0.3, 0.7)])
def test_clr_table_is_torchs(lr, lr_decay):
    from rl_ctr_prediction_b200.tables import AdagradSchedule
    s = AdagradSchedule(lr, lr_decay, "cpu", length=64)
    assert s.tensor.dtype == torch.float32 and s.length >= 64
    assert torch.equal(s.tensor[1:41], _torch_clr(lr, lr_decay, 40)[1:])
    ref = torch.tensor([lr / (1 + (t - 1) * lr_decay) for t in range(1, 41)], dtype=torch.float64).to(torch.float32)
    assert torch.equal(s.tensor[1:41], ref)
    s.set_lr(lr * 1.7, 13)                            # an lr edit before step 13: earlier steps keep the lr they ran with
    assert torch.equal(s.tensor[1:41], _torch_clr(lr, lr_decay, 40, edit=(13, lr * 1.7))[1:])
    s.ensure(5000)                                    # a longer table keeps the edited entries
    assert torch.equal(s.tensor[1:41], _torch_clr(lr, lr_decay, 40, edit=(13, lr * 1.7))[1:])
    assert float(s.tensor[4000]) == float(torch.tensor(lr * 1.7 / (1 + 3999 * lr_decay), dtype=torch.float64).float())


def test_constructor_validates_like_torch():
    from rl_ctr_prediction_b200 import optim
    p = [torch.nn.Parameter(torch.zeros(3))]
    for kw, msg in ((dict(lr=-1e-3), "Invalid learning rate"), (dict(lr_decay=-1.0), "Invalid lr_decay value"),
                    (dict(weight_decay=-1e-5), "Invalid weight_decay value"),
                    (dict(initial_accumulator_value=-0.1), "Invalid initial_accumulator_value value"),
                    (dict(eps=-1e-10), "Invalid epsilon value")):
        with pytest.raises(ValueError, match=msg):
            torch.optim.Adagrad(p, **kw)
        with pytest.raises(ValueError, match=msg):
            optim.Adagrad(p, **kw)
    with pytest.raises(ValueError, match="empty parameter list"):
        optim.Adagrad([])
    with pytest.raises(ValueError, match="eps == 0 with initial_accumulator_value == 0"):
        optim.Adagrad(p, eps=0.0)
    with pytest.raises(ValueError, match="Invalid mode"):
        optim.Adagrad(p, mode="sparse")
    optim.Adagrad(p, eps=0.0, initial_accumulator_value=0.1)          # either one positive is enough
    o = optim.Adagrad(p)
    ref = torch.optim.Adagrad(p).param_groups[0]
    for k in ("lr", "lr_decay", "weight_decay", "initial_accumulator_value", "eps"):
        assert o.param_groups[0][k] == ref[k], k                      # torch's defaults
    o.param_groups[0]["eps"] = 1e-8
    with pytest.raises(_lib.RlctrError, match="changing eps after construction"):
        o._sync_hyper()
    o.param_groups[0]["eps"] = 1e-10
    o.param_groups[0]["lr"] = 0.5                                     # lr may change
    o._sync_hyper()
    assert o.lr == 0.5
