"""Parity of every C-ABI entry point (include/rlctr.h) against the CPU oracle and the golden vectors
produced by the real reference modules.  Calls go through ctypes into librlctr_sm100a.so.

Bars (BASELINE.json north_star): gathered rows bit-exact; logits, loss, gradients, Adam state and
policy log-probs within 1e-5 relative in fp32 (RTOL below; ATOL covers values near zero).
"""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import state_from_golden
from oracle import np_oracle as O

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-5, 1e-6
DEV = "cuda:0"


@pytest.fixture(scope="module")
def lib():
    from rl_ctr_prediction_b200 import _lib
    return _lib.load()


def L():
    from rl_ctr_prediction_b200 import _lib
    return _lib


def T():
    from rl_ctr_prediction_b200 import tables
    return tables


def close(a, b, rtol=RTOL, atol=None):
    """|a - b| <= rtol * max(|b|, scale): the north star's "1e-5 relative in fp32" read against the
    SCALE of the quantity (scale = max |b| over the array) -- a logit or a gradient is a sum of terms
    that cancel, so two correct fp32 evaluations (e.g. torch on CPU vs torch on GPU) differ by
    ~1e-7 * scale in absolute terms however small the individual result is.  An explicit `atol`
    overrides the scale term."""
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    b = b.detach().cpu().numpy() if isinstance(b, torch.Tensor) else np.asarray(b)
    a, b = a.astype(np.float64), b.astype(np.float64)
    if atol is None:
        atol = rtol * (np.abs(b).max() if b.size else 0.0)
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol)


def fused_fm_table(lin, emb):
    """[N, round4(1+D)] = [w | v | pad]"""
    N, D = emb.shape
    g = T().Geometry.fm(N, D)
    tab = torch.zeros(N, g.row_stride)
    tab[:, 0:1] = torch.as_tensor(lin).reshape(N, 1)
    tab[:, 1:1 + D] = torch.as_tensor(emb)
    return tab.to(DEV), g


def fused_ffm_table(lin, tables):
    Fn, N, D = tables.shape
    g = T().Geometry.ffm(N, Fn, D)
    tab = torch.zeros(N, g.row_stride)
    for t in range(Fn):
        tab[:, t * D:(t + 1) * D] = torch.as_tensor(tables[t])
    tab[:, g.lin_col] = torch.as_tensor(lin).reshape(N)
    return tab.to(DEV), g


_KEEP = []      # device tensors whose raw pointers were handed to the library: keep them alive until the test ends


@pytest.fixture(autouse=True)
def _keepalive():
    yield
    torch.cuda.synchronize()
    _KEEP.clear()


def dev(x, dtype=None):
    if x is None:
        return None
    t = torch.as_tensor(np.ascontiguousarray(x))
    if dtype is not None:
        t = t.to(dtype)
    t = t.to(DEV).contiguous()
    _KEEP.append(t)
    return t


def st():
    return L().stream()


def rng_case(seed, B, F, N, D, zipf=True, scale=0.3):
    rng = np.random.default_rng(seed)
    if zipf:
        per = max(N // F, 1)
        ids = np.stack([np.minimum(rng.zipf(1.3, size=B) - 1, per - 1) + f * per for f in range(F)], axis=1)
        ids = np.minimum(ids, N - 1)
    else:
        ids = rng.integers(0, N, size=(B, F))
    emb = (rng.standard_normal((N, D)) * scale).astype(np.float32)
    lin = (rng.standard_normal((N, 1)) * scale).astype(np.float32)
    bias = np.array([0.1], dtype=np.float32)
    y = (rng.random(B) < 0.3).astype(np.int64)
    return ids.astype(np.int64), emb, lin, bias, y


# ------------------------------------------------------------------------------------------------
# K1 forward
# ------------------------------------------------------------------------------------------------
def run_embed_fwd(lib, ids, tab, g, bias, fm=True, want_rows=True, want_sums=True):
    B, F = ids.shape
    ids_d = dev(ids)
    logit = torch.empty(B, device=DEV)
    pctr = torch.empty(B, device=DEV)
    sums = torch.empty(B, g.row_stride, device=DEV) if want_sums else None
    rows = torch.empty(B, F * g.dim, device=DEV) if want_rows else None
    t = T().table_struct(tab, g)
    rc = lib.rlctr_embed_fwd(L().ptr(ids_d), C.byref(t), L().ptr(dev(bias)), L().ptr(logit), L().ptr(pctr), 1,
                             L().ptr(sums), L().ptr(rows), 0, B, F, 1 if fm else 0, st())
    assert rc == 0, L().load().rlctr_strerror(rc)
    torch.cuda.synchronize()
    return logit, pctr, sums, rows


@pytest.mark.parametrize("D", [10, 8, 16, 4, 2])
@pytest.mark.parametrize("B,F", [(1, 15), (37, 15), (1000, 15), (64, 3), (50, 33)])
def test_embed_fwd_fm(lib, B, F, D):
    ids, emb, lin, bias, _ = rng_case(B * 131 + D, B, F, 997, D)
    tab, g = fused_fm_table(lin, emb)
    logit, pctr, sums, rows = run_embed_fwd(lib, ids, tab, g, bias)
    # gathered rows: bit-exact
    assert np.array_equal(rows.cpu().numpy().reshape(B, F, D), emb[ids])
    close(logit, O.fm_logit(ids, emb, lin, bias).reshape(-1))
    close(logit, O.fm_logit(ids, emb, lin, bias, np.float64).reshape(-1))
    close(pctr, O.sigmoid(O.fm_logit(ids, emb, lin, bias)).reshape(-1))
    close(sums[:, 1:1 + D], emb[ids].sum(axis=1))


def test_embed_fwd_golden_kat(lib, golden):
    x = golden["kat/x"]
    sd = state_from_golden(golden, "kat/FM/init")
    tab, g = fused_fm_table(sd["linear.weight"], sd["feature_embedding.weight"])
    _, pctr, _, _ = run_embed_fwd(lib, x, tab, g, sd["bias"])
    close(pctr, golden["kat/FM/pctr"].reshape(-1))
    # LR on the fused table (no FM term) and on the scalar table
    sd = state_from_golden(golden, "kat/LR/init")
    tab, g = fused_fm_table(sd["linear.weight"], np.zeros((64, 10), np.float32))
    _, pctr, _, _ = run_embed_fwd(lib, x, tab, g, sd["bias"], fm=False)
    close(pctr, golden["kat/LR/pctr"].reshape(-1))
    g1 = T().Geometry.lr(64)
    tab1 = dev(sd["linear.weight"].reshape(-1))
    _, pctr, _, _ = run_embed_fwd(lib, x, tab1, g1, sd["bias"], fm=False, want_rows=False, want_sums=False)
    close(pctr, golden["kat/LR/pctr"].reshape(-1))


def test_embed_fwd_hand_kat(lib):
    # SURVEY section 4: F=2, D=2, v1=(1,2), v2=(3,4): 0.5*sum_d[(sum v)^2 - sum v^2] = 11
    emb = np.array([[1, 2], [3, 4]], np.float32)
    lin = np.zeros((2, 1), np.float32)
    tab, g = fused_fm_table(lin, emb)
    logit, _, _, _ = run_embed_fwd(lib, np.array([[0, 1]]), tab, g, np.zeros(1, np.float32))
    assert logit.item() == 11.0


def test_embed_fwd_saturation_and_oob(lib):
    # default N(0,1) init saturates fp32 sigmoid to exactly 0/1 (SURVEY N2); out-of-range id = zero row
    ids, emb, lin, bias, _ = rng_case(5, 256, 15, 500, 10, scale=1.0)
    tab, g = fused_fm_table(lin, emb)
    _, pctr, _, _ = run_embed_fwd(lib, ids, tab, g, bias)
    ref = O.sigmoid(O.fm_logit(ids, emb, lin, bias)).reshape(-1)
    close(pctr, ref)
    p = pctr.cpu().numpy()
    assert ((p == 0) | (p == 1)).sum() == ((ref == 0) | (ref == 1)).sum() > 0
    ids2 = ids.copy()
    ids2[:, 3] = 10 ** 9
    emb0 = np.vstack([emb, np.zeros((1, 10), np.float32)])
    lin0 = np.vstack([lin, np.zeros((1, 1), np.float32)])
    ids_ref = ids2.copy()
    ids_ref[:, 3] = 500
    logit, _, _, _ = run_embed_fwd(lib, ids2, tab, g, bias)
    close(logit, O.fm_logit(ids_ref, emb0, lin0, bias).reshape(-1))


def test_embed_fwd_empty_and_errors(lib):
    ids, emb, lin, bias, _ = rng_case(1, 4, 15, 100, 10)
    tab, g = fused_fm_table(lin, emb)
    t = T().table_struct(tab, g)
    assert lib.rlctr_embed_fwd(L().ptr(dev(ids)), C.byref(t), None, None, None, 1, None, None, 0, 0, 15, 1, st()) == 0
    # ids == NULL means sample-ordered rows: the table must then hold batch * fields of them (100 < 7 * 15)
    assert lib.rlctr_embed_fwd(None, C.byref(t), None, None, None, 1, None, None, 0, 7, 15, 1, st()) == -1
    bad = L().Table(L().ptr(tab), 100, 10, 0, 1, 9)          # stride not a multiple of 4
    assert lib.rlctr_embed_fwd(L().ptr(dev(ids)), C.byref(bad), None, None, None, 1, None, None, 0, 4, 15, 1, st()) == -2


def test_gather_rows_bit_exact(lib):
    ids, emb, lin, _, _ = rng_case(9, 5000, 15, 30000, 10, zipf=False)
    tab, g = fused_fm_table(lin, emb)
    flat = dev(ids.reshape(-1))
    out = torch.empty(flat.numel(), g.row_stride, device=DEV)
    t = T().table_struct(tab, g)
    assert lib.rlctr_gather_rows(L().ptr(flat), flat.numel(), C.byref(t), L().ptr(out), st()) == 0
    assert torch.equal(out, tab[flat])


# ------------------------------------------------------------------------------------------------
# K2 FFM
# ------------------------------------------------------------------------------------------------
def run_ffm(lib, ids, tab, g, bias, D, partners=False):
    B, F = ids.shape
    logit = torch.empty(B, device=DEV)
    pctr = torch.empty(B, device=DEV)
    part = torch.empty(B * F, g.row_stride, device=DEV) if partners else None
    t = T().table_struct(tab, g)
    rc = lib.rlctr_ffm_fwd(L().ptr(dev(ids)), C.byref(t), L().ptr(dev(bias)), L().ptr(logit), L().ptr(pctr), 1,
                           L().ptr(part), B, F, D, st())
    assert rc == 0, rc
    torch.cuda.synchronize()
    return logit, pctr, part


@pytest.mark.parametrize("B,F,D", [(1, 15, 10), (77, 15, 10), (300, 15, 8), (40, 4, 3), (16, 22, 4)])
def test_ffm_fwd(lib, B, F, D):
    rng = np.random.default_rng(B + F + D)
    N = 211
    ids = rng.integers(0, N, size=(B, F)).astype(np.int64)
    tables = (rng.standard_normal((F, N, D)) * 0.3).astype(np.float32)
    lin = (rng.standard_normal((N, 1)) * 0.3).astype(np.float32)
    bias = np.array([-0.2], np.float32)
    tab, g = fused_ffm_table(lin, tables)
    logit, pctr, part = run_ffm(lib, ids, tab, g, bias, D, partners=True)
    close(logit, O.ffm_logit(ids, tables, lin, bias, np.float64).reshape(-1))
    close(pctr, O.sigmoid(O.ffm_logit(ids, tables, lin, bias)).reshape(-1))
    # partner rows == d logit / d row: G[t, b, f] of the oracle with dz = 1, plus 1 at the linear col
    G = O.ffm_row_grads(np.ones(B, np.float32), ids, tables)          # [F_table, B, F_field, D]
    part = part.cpu().numpy().reshape(B, F, g.row_stride)
    for t in range(F):
        assert np.array_equal(part[:, :, t * D:(t + 1) * D], G[t])
    assert np.all(part[:, :, g.lin_col] == 1.0)
    assert np.all(part[:, :, g.lin_col + 1:] == 0.0)


def test_ffm_golden_kat(lib, golden):
    sd = state_from_golden(golden, "kat/FFM/init")
    tables = np.stack([sd[f"field_feature_embeddings.{t}.weight"] for t in range(15)])
    tab, g = fused_ffm_table(sd["linear.weight"], tables)
    _, pctr, _ = run_ffm(lib, golden["kat/x"], tab, g, sd["bias"], 10)
    close(pctr, golden["kat/FFM/pctr"].reshape(-1))


# ------------------------------------------------------------------------------------------------
# K5 Feature_Embedding
# ------------------------------------------------------------------------------------------------
def test_featemb_golden(lib, golden):
    for wkey, xkey, okey in (("kat/FE/weight", "kat/x", "kat/FE/out"), ("fe/weight", "fe/x", "fe/out")):
        w, x, ref = golden[wkey], golden[xkey], golden[okey]
        N, D = w.shape
        g = T().Geometry.fm(N, D, with_linear=False)
        tab = torch.zeros(N, g.row_stride)
        tab[:, :D] = torch.as_tensor(w)
        tab = tab.to(DEV)
        B, F = x.shape
        out = torch.empty(B, ref.shape[1], device=DEV)
        t = T().table_struct(tab, g)
        assert lib.rlctr_featemb_fwd(L().ptr(dev(x)), C.byref(t), L().ptr(out), out.stride(0), B, F, st()) == 0
        close(out, ref)
        # the flattened rows are a bit-exact copy
        assert np.array_equal(out[:, F * (F - 1) // 2:].cpu().numpy(), w[x].reshape(B, -1))
        close(out, O.feature_embedding(x, w))


# ------------------------------------------------------------------------------------------------
# loss head
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [1, 48, 4096, 300001])
def test_bce_fwd_bwd(lib, B):
    rng = np.random.default_rng(B)
    z = (rng.standard_normal(B) * 30).astype(np.float32)       # deep into the saturated regime (N2)
    y = (rng.random(B) < 0.4).astype(np.int64)
    ws = torch.zeros(L().RLCTR_REDUCE_WS_BYTES, dtype=torch.uint8, device=DEV)
    pctr = torch.empty(B, device=DEV)
    loss = torch.empty(1, device=DEV)
    dz = torch.empty(B, device=DEV)
    db = torch.empty(1, device=DEV)
    for yi, yf in ((dev(y), None), (None, dev(y, torch.float32))):
        rc = lib.rlctr_bce_fwd_bwd(L().ptr(dev(z)), L().ptr(yi), L().ptr(yf), L().ptr(pctr), L().ptr(loss), L().ptr(dz),
                                   L().ptr(db), L().ptr(ws), B, st())
        assert rc == 0
        p_ref, l_ref, dz_ref = O.loss_head(z, y)
        close(pctr, p_ref.reshape(-1))
        close(loss, l_ref, rtol=1e-5)
        close(dz, dz_ref.reshape(-1), atol=1e-12)
        close(db, dz_ref.astype(np.float64).sum(), rtol=1e-4, atol=1e-7)
    # and against torch's own CPU autograd (the op the reference calls)
    zt = torch.tensor(z, requires_grad=True)
    lt = torch.nn.BCELoss()(torch.sigmoid(zt).view(-1, 1), torch.tensor(y).float().view(-1, 1))
    lt.backward()
    close(loss, lt.item(), rtol=1e-5)
    close(dz, zt.grad, atol=1e-12)
    # determinism: fixed-shape tree
    l1 = loss.clone()
    lib.rlctr_bce_fwd_bwd(L().ptr(dev(z)), L().ptr(dev(y)), None, L().ptr(pctr), L().ptr(loss), L().ptr(dz),
                          L().ptr(db), L().ptr(ws), B, st())
    assert torch.equal(l1, loss)


def test_sigmoid_bwd(lib):
    B = 1000
    rng = np.random.default_rng(0)
    p = rng.random(B).astype(np.float32)
    g = rng.standard_normal(B).astype(np.float32)
    ws = torch.zeros(L().RLCTR_REDUCE_WS_BYTES, dtype=torch.uint8, device=DEV)
    dz = torch.empty(B, device=DEV)
    db = torch.empty(1, device=DEV)
    assert lib.rlctr_sigmoid_bwd(L().ptr(dev(g)), L().ptr(dev(p)), L().ptr(dz), L().ptr(db), L().ptr(ws), B, st()) == 0
    ref = g * (np.float32(1) - p) * p
    close(dz, ref, atol=1e-9)
    close(db, ref.astype(np.float64).sum(), rtol=1e-5)


# ------------------------------------------------------------------------------------------------
# K3 sort + segment-reduce + Adam
# ------------------------------------------------------------------------------------------------
def do_sort(lib, ids_flat_d, n_rows):
    n = ids_flat_d.numel()
    sid = torch.empty(n, dtype=torch.int32, device=DEV)
    ss = torch.empty(n, dtype=torch.int32, device=DEV)
    wsb = lib.rlctr_sort_ws_bytes(n, n_rows)
    ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
    assert lib.rlctr_sort_ids(L().ptr(ids_flat_d), n, n_rows, L().ptr(sid), L().ptr(ss), L().ptr(ws), wsb, st()) == 0
    return sid, ss


@pytest.mark.parametrize("n,n_rows", [(1, 10), (720, 255), (100000, 1000), (983040, 10_000_000)])
def test_sort_ids_stable(lib, n, n_rows):
    rng = np.random.default_rng(n)
    ids = rng.integers(0, n_rows, size=n).astype(np.int64)
    sid, ss = do_sort(lib, dev(ids), n_rows)
    order = np.argsort(ids, kind="stable")
    assert np.array_equal(sid.cpu().numpy().astype(np.int64), ids[order])
    assert np.array_equal(ss.cpu().numpy().astype(np.int64), order)


def adam_struct(m, v, stamp, sched, step, wd=1e-5):
    return L().Adam(L().ptr(m), L().ptr(v), L().ptr(stamp), L().ptr(sched), L().ptr(step), sched.shape[0], -1, 0.9, 0.999,
                    1e-8, wd)


def make_sched(lr, n=64):
    return T().AdamSchedule(lr, (0.9, 0.999), torch.device(DEV), n).tensor


@pytest.mark.parametrize("D", [10, 8, 16])
@pytest.mark.parametrize("zipf", [True, False])
def test_rows_grad_dense_fm(lib, D, zipf):
    """embedding_dense_backward parity: FM row gradients scattered into a dense [N, rs] gradient."""
    B, F, N = 600, 15, 400
    ids, emb, lin, bias, y = rng_case(D + 100 * zipf, B, F, N, D, zipf=zipf)
    if zipf:
        ids[:, 0] = 0                       # one id hit by every sample: the long-run path (> LONG_RUN)
        ids[0, 1] = ids[0, 0]               # repeated id inside one sample
    tab, g = fused_fm_table(lin, emb)
    logit, _, sums, _ = run_embed_fwd(lib, ids, tab, g, bias, want_rows=False)
    _, _, dz_ref = O.loss_head(logit.cpu().numpy(), y)
    dz = dev(dz_ref.reshape(-1))
    sid, ss = do_sort(lib, dev(ids.reshape(-1)), N)
    dense = torch.zeros(N, g.row_stride, device=DEV)
    grad = L().RowGrad(None, L().ptr(dz), L().ptr(sums), None, F, 0)
    t = T().table_struct(tab, g)
    wsb = lib.rlctr_rows_ws_bytes(B * F)
    ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
    assert lib.rlctr_rows_grad_dense(L().ptr(sid), L().ptr(ss), B * F, C.byref(grad), C.byref(t), L().ptr(dense),
                                     L().ptr(ws), wsb, st()) == 0
    demb, dlin = O.fm_row_grads(dz_ref, ids, emb)
    ref_emb = O.scatter_dense(ids, demb, N, np.float64)
    ref_lin = O.scatter_dense(ids, dlin.reshape(B, F, 1), N, np.float64)
    close(dense[:, 1:1 + D], ref_emb, rtol=2e-5)
    close(dense[:, 0:1], ref_lin, rtol=2e-5)
    # bit-identical from run to run (no atomics on the data path)
    dense2 = torch.zeros_like(dense)
    lib.rlctr_rows_grad_dense(L().ptr(sid), L().ptr(ss), B * F, C.byref(grad), C.byref(t), L().ptr(dense2),
                              L().ptr(ws), wsb, st())
    assert torch.equal(dense, dense2)


def test_rows_grad_golden_fm(lib, golden):
    """dense gradient of step 0 of the golden FM trajectory == autograd of the real reference."""
    for case in ("train", "sat"):
        sd = state_from_golden(golden, f"{case}/FM/init")
        x, y = golden["train/x"][0], golden["train/y"][0]
        N = 255
        tab, g = fused_fm_table(sd["linear.weight"], sd["feature_embedding.weight"])
        B, F = x.shape
        logit, _, sums, _ = run_embed_fwd(lib, x, tab, g, sd["bias"], want_rows=False)
        ws0 = torch.zeros(L().RLCTR_REDUCE_WS_BYTES, dtype=torch.uint8, device=DEV)
        dz = torch.empty(B, device=DEV)
        loss = torch.empty(1, device=DEV)
        assert lib.rlctr_bce_fwd_bwd(L().ptr(logit), L().ptr(dev(y)), None, None, L().ptr(loss), L().ptr(dz), None,
                                     L().ptr(ws0), B, st()) == 0
        close(loss, golden[f"{case}/FM/loss0"])
        sid, ss = do_sort(lib, dev(x.reshape(-1)), N)
        dense = torch.zeros(N, g.row_stride, device=DEV)
        grad = L().RowGrad(None, L().ptr(dz), L().ptr(sums), None, F, 0)
        t = T().table_struct(tab, g)
        wsb = lib.rlctr_rows_ws_bytes(B * F)
        ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
        assert lib.rlctr_rows_grad_dense(L().ptr(sid), L().ptr(ss), B * F, C.byref(grad), C.byref(t), L().ptr(dense),
                                         L().ptr(ws), wsb, st()) == 0
        close(dense[:, 1:11], golden[f"{case}/FM/grad0/feature_embedding.weight"], rtol=2e-5)
        close(dense[:, 0:1], golden[f"{case}/FM/grad0/linear.weight"], rtol=2e-5)


@pytest.mark.parametrize("mode", ["lazy", "dense"])
def test_rows_adam_matches_dense_adam(lib, mode):
    """K3 + lazy replay == the reference's dense Adam with L2 over EVERY row (SURVEY N3), 4 steps."""
    B, F, N, D, STEPS, lr, wd = 64, 15, 300, 10, 4, 1e-3, 1e-5
    ids0, emb, lin, bias, _ = rng_case(77, B, F, N, D)
    tab, g = fused_fm_table(lin, emb)
    rs = g.row_stride
    m = torch.zeros_like(tab)
    v = torch.zeros_like(tab)
    stamp = torch.zeros(N, dtype=torch.int32, device=DEV)
    step = torch.zeros(1, dtype=torch.int32, device=DEV)
    sched = make_sched(lr)
    a = adam_struct(m, v, stamp, sched, step, wd)
    t = T().table_struct(tab, g)
    # oracle state (padded layout, pad columns stay 0)
    P = tab.cpu().numpy().copy()
    Mo, Vo = np.zeros_like(P), np.zeros_like(P)
    rng = np.random.default_rng(3)
    for s in range(1, STEPS + 1):
        ids = rng.integers(0, N // 3, size=(B, F)).astype(np.int64) + (s % 3) * (N // 3)   # rows go stale and come back
        dzv = (rng.standard_normal(B) * 0.01).astype(np.float32)
        staged = (rng.standard_normal((B * F, rs)) * 0.01).astype(np.float32)
        staged[:, 1 + D:] = 0
        sid, ss = do_sort(lib, dev(ids.reshape(-1)), N)
        if mode == "lazy":
            assert lib.rlctr_rows_catchup(L().ptr(sid), B * F, C.byref(t), C.byref(a), st()) == 0
            # rows of this batch now equal the dense-Adam state after s-1 steps
            got = tab.cpu().numpy()
            uniq = np.unique(ids)
            close(got[uniq], P[uniq], rtol=2e-5, atol=1e-7)
        grad = L().RowGrad(L().ptr(dev(staged)), L().ptr(dev(dzv)), None, None, F, 0)
        wsb = lib.rlctr_rows_ws_bytes(B * F)
        ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
        assert lib.rlctr_rows_adam(L().ptr(sid), L().ptr(ss), B * F, C.byref(grad), C.byref(t), C.byref(a), L().ptr(ws),
                                   wsb, st()) == 0
        assert lib.rlctr_step_advance(L().ptr(step), 1, st()) == 0
        if mode == "dense":
            assert lib.rlctr_adam_flush(C.byref(t), C.byref(a), 0, N, st()) == 0
        # oracle: dense gradient = scatter(staged) + dz at the linear column, Adam over ALL rows
        G = O.scatter_dense(ids, staged.reshape(B, F, rs), N)
        G[:, 0] += O.scatter_dense(ids, np.repeat(dzv, F).reshape(B, F, 1), N)[:, 0]
        P, Mo, Vo = O.adam_step(P, G, Mo, Vo, s, lr, wd)
        P[:, 1 + D:] = 0
    assert lib.rlctr_adam_flush(C.byref(t), C.byref(a), 0, N, st()) == 0
    torch.cuda.synchronize()
    assert step.item() == STEPS and int(stamp.min()) == STEPS
    close(tab, P, rtol=2e-5, atol=1e-7)
    close(m, Mo, rtol=2e-5, atol=1e-9)
    close(v, Vo, rtol=2e-5, atol=1e-12)



@pytest.mark.parametrize("kind,D", [("fm", 10), ("fm", 8), ("fm", 2), ("lr", 0)])
@pytest.mark.parametrize("heavy", [False, True])
def test_rows_lookup_stage_update_equals_dense_adam(lib, kind, D, heavy):
    """rlctr_rows_lookup (read once, replay in registers, stage + push to the samples) -> streamed forward rows ->
    rlctr_rows_adam reading the stage == the reference's dense Adam with L2 over EVERY row (SURVEY N3).  The table keeps the
    [row | exp_avg | exp_avg_sq] records with the stamp inside; ids go stale for several steps and come back; `heavy` adds an
    id with hundreds of occurrences (the block-per-run kernels)."""
    from rl_ctr_prediction_b200.tables import Geometry, TableAdamState, table_struct
    B, F, N, STEPS, lr, wd = 96, 15, 600, 7, 1e-3, 1e-5
    rng = np.random.default_rng(11 + D)
    g = (Geometry.lr(N) if kind == "lr" else Geometry.fm(N, D)).with_state()
    rs, used = g.row_stride, g.used
    tab = torch.zeros(N, g.row_pitch, device=DEV)
    tab[:, :used] = torch.as_tensor((rng.standard_normal((N, used)) * 0.3).astype(np.float32)).to(DEV)
    opt = TableAdamState(tab, g, lr, (0.9, 0.999), 1e-8, wd, "lazy")
    assert opt.lookup_ok and opt.stamp_col >= 0
    P = np.zeros((N, rs), np.float32)
    P[:, :used] = tab[:, :used].cpu().numpy()
    Mo, Vo = np.zeros_like(P), np.zeros_like(P)
    t = table_struct(tab, g)
    n = B * F
    sf = lib.rlctr_lookup_stage_floats(C.byref(t))
    assert sf == (4 if kind == "lr" else 3 * ((used + 3) // 4 * 4))
    for s in range(1, STEPS + 1):
        ids = rng.integers(0, N // 3, size=(B, F)).astype(np.int64) + (s % 3) * (N // 3)
        if heavy:
            ids[rng.random((B, F)) < 0.4] = (s % 3) * (N // 3) + 5         # one id with ~570 occurrences
        ids[0, 0] = N + 7                                                   # out of range: all-zero row, no update
        dzv = (rng.standard_normal(B) * 0.01).astype(np.float32)
        sid, ss = do_sort(lib, dev(ids.reshape(-1)), N)
        stage = torch.full((n * sf,), float("nan"), device=DEV)
        gathered = torch.zeros(n, rs, device=DEV)
        a = opt.struct()
        lk = L().Lookup(stage.data_ptr(), 0, 0)
        lk.gathered[0] = gathered.data_ptr()
        wsb = lib.rlctr_rows_ws_bytes(n)
        ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
        rc = lib.rlctr_rows_lookup(L().ptr(sid), L().ptr(ss), n, C.byref(t), C.byref(a), C.byref(lk), L().ptr(ws), wsb, st())
        assert rc == 0, lib.rlctr_strerror(rc)
        # every sample's row == the dense-Adam state after s-1 steps (out-of-range id: zeros); padding columns clean
        want = np.zeros((n, rs), np.float32)
        flat = ids.reshape(-1)
        ok = flat < N
        want[ok] = P[flat[ok]]
        got = gathered.cpu().numpy()
        close(got[:, :used], want[:, :used], rtol=2e-5, atol=1e-7)
        assert not got[:, used:].any()
        # gradient: dz at the linear column (+ dz * (S - v) on the latent columns for the FM rows)
        sums = None
        if kind == "fm":
            S = got.reshape(B, F, rs).sum(axis=1)
            sums = dev(S)
        grad = L().RowGrad(None, L().ptr(dev(dzv)), L().ptr(sums), None, F, 0)
        a2 = opt.struct(stage)
        assert lib.rlctr_rows_adam(L().ptr(sid), L().ptr(ss), n, C.byref(grad), C.byref(t), C.byref(a2), L().ptr(ws), wsb,
                                   st()) == 0
        assert lib.rlctr_step_advance(L().ptr(opt.step), 1, st()) == 0
        opt.dirty = True
        G = np.zeros((N, rs), np.float64)
        rows64 = want.reshape(B, F, rs).astype(np.float64)
        S64 = rows64.sum(axis=1)
        for b in range(B):
            for f in range(F):
                i = ids[b, f]
                if i >= N:
                    continue
                G[i, 0] += dzv[b]
                if kind == "fm":
                    G[i, 1:1 + D] += np.float64(dzv[b]) * (S64[b, 1:1 + D] - rows64[b, f, 1:1 + D])
        P, Mo, Vo = O.adam_step(P, G.astype(np.float32), Mo, Vo, s, lr, wd)
        P[:, used:] = 0
    opt.flush(tab)
    torch.cuda.synchronize()
    rec = tab.cpu().numpy()
    close(rec[:, :used], P[:, :used], rtol=2e-5, atol=1e-7)
    if kind == "lr":                  # moments: 2e-5 of their scale (the oracle sums the occurrences' gradients in fp64)
        close(rec[:, 1], Mo[:, 0], rtol=2e-5)
        close(rec[:, 2], Vo[:, 0], rtol=2e-5)
    else:
        close(rec[:, rs:rs + used], Mo[:, :used], rtol=2e-5)
        close(rec[:, 2 * rs:2 * rs + used], Vo[:, :used], rtol=2e-5)
    assert (tab[:, opt.stamp_col].view(torch.int32) == STEPS).all()


def test_embed_fwd_streamed_rows_equal_gather_by_id(lib):
    """rlctr_embed_fwd with ids == NULL over sample-ordered rows == the same call gathering by id (bit for bit)."""
    B, F, N, D = 333, 15, 5000, 10
    ids, emb, lin, bias, _ = rng_case(5, B, F, N, D)
    tab, g = fused_fm_table(lin, emb)
    z0, p0, s0, r0 = run_embed_fwd(lib, ids, tab, g, bias)
    rows = tab[torch.as_tensor(ids.reshape(-1)).to(DEV)].contiguous()
    t = L().Table(rows.data_ptr(), B * F, g.row_stride, g.lin_col, g.emb_col, g.dim, g.row_stride)
    logit, pctr = torch.empty(B, device=DEV), torch.empty(B, device=DEV)
    sums, out = torch.empty(B, g.row_stride, device=DEV), torch.empty(B, F * D, device=DEV)
    assert lib.rlctr_embed_fwd(None, C.byref(t), L().ptr(dev(bias)), L().ptr(logit), L().ptr(pctr), 1, L().ptr(sums),
                               L().ptr(out), 0, B, F, 1, st()) == 0
    torch.cuda.synchronize()
    assert torch.equal(logit, z0) and torch.equal(pctr, p0) and torch.equal(sums, s0) and torch.equal(out, r0)
    t.n_rows = B * F - 1                                  # fewer rows than samples x fields: refused
    assert lib.rlctr_embed_fwd(None, C.byref(t), None, L().ptr(logit), None, 1, None, None, 0, B, F, 1, st()) == -1


def test_dense_adam(lib):
    n, lr, wd = 12345, 1e-3, 1e-5
    rng = np.random.default_rng(5)
    p = rng.standard_normal(n).astype(np.float32)
    P, Mo, Vo = p.copy(), np.zeros(n, np.float32), np.zeros(n, np.float32)
    pd_, m, v = dev(p), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    step = torch.zeros(1, dtype=torch.int32, device=DEV)
    sched = make_sched(lr)
    pt = torch.tensor(p.copy(), requires_grad=True)
    topt = torch.optim.Adam([pt], lr=lr, weight_decay=wd)
    for s in range(1, 4):
        gnp = rng.standard_normal(n).astype(np.float32)
        assert lib.rlctr_dense_adam(L().ptr(pd_), L().ptr(dev(gnp)), L().ptr(m), L().ptr(v), n, L().ptr(sched),
                                    L().ptr(step), 0.9, 0.999, 1e-8, wd, st()) == 0
        assert lib.rlctr_step_advance(L().ptr(step), 1, st()) == 0
        P, Mo, Vo = O.adam_step(P, gnp, Mo, Vo, s, lr, wd)
        pt.grad = torch.tensor(gnp)
        topt.step()
    close(pd_, P, rtol=2e-6)
    close(pd_, pt.detach(), rtol=2e-6)           # torch.optim.Adam itself (CPU)


# ------------------------------------------------------------------------------------------------
# K6 generate_preds, REINFORCE head
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M", [3, 5, 6])
def test_generate_preds_golden(lib, golden, M):
    pre = f"gp/v0_M{M}/"
    pctr, w, lab = golden[pre + "pctr"], golden[pre + "w"], golden[pre + "label"]
    B = pctr.shape[0]
    for variant, akey in ((0, pre + "action"), (1, f"gp/v1_M{M}/action")):
        act = golden[akey]
        y = torch.empty(B, device=DEV)
        wo = torch.empty(B, M, device=DEV)
        r = torch.empty(B, device=DEV)
        assert lib.rlctr_generate_preds(L().ptr(dev(pctr)), L().ptr(dev(w)), L().ptr(dev(act.reshape(-1))),
                                        L().ptr(dev(lab.reshape(-1))), L().ptr(y), L().ptr(wo), L().ptr(r), B, M, variant,
                                        st()) == 0
        vpre = pre if variant == 0 else f"gp/v1_M{M}/"
        close(y, golden[vpre + "y"].reshape(-1), rtol=1e-5, atol=1e-7)
        assert np.array_equal(r.cpu().numpy(), golden[vpre + "reward"].reshape(-1))
        if variant == 0:
            close(wo, golden[pre + "w_out"], rtol=1e-5, atol=1e-7)


def test_generate_preds_random_vs_oracle(lib):
    rng = np.random.default_rng(11)
    for M in (2, 3, 8):
        B = 5000
        pctr = rng.random((B, M)).astype(np.float32)
        w = O.softmax(rng.standard_normal((B, M)).astype(np.float32) * 2)
        lab = (rng.random(B) < 0.5).astype(np.int64)
        for variant, lo in ((0, 2), (1, 1)):
            act = rng.integers(lo, M + 1, size=B).astype(np.int64)
            act[:7] = 0                                            # no branch matches: y = r = 1 (main.py:185-186)
            y = torch.empty(B, device=DEV)
            wo = torch.empty(B, M, device=DEV)
            r = torch.empty(B, device=DEV)
            assert lib.rlctr_generate_preds(L().ptr(dev(pctr)), L().ptr(dev(w)), L().ptr(dev(act)), L().ptr(dev(lab)),
                                            L().ptr(y), L().ptr(wo), L().ptr(r), B, M, variant, st()) == 0
            yo, wo_o, ro = O.generate_preds(pctr, w, act, lab, variant)
            close(y, yo.reshape(-1), rtol=1e-5, atol=1e-7)
            close(wo, wo_o, rtol=1e-5, atol=1e-7)
            # rewards compare y with the baseline: allow flips only where they are within rounding of each other
            mism = r.cpu().numpy() != ro.reshape(-1)
            assert mism.mean() < 1e-3


def _gp10(lib, pctr, w, c, act, lab):
    B, M = pctr.shape
    y = torch.empty(B, device=DEV)
    co = torch.empty(B, M, device=DEV)
    r = torch.empty(B, device=DEV)
    wsb = lib.rlctr_generate_preds_v10_ws_bytes(B)
    ws = torch.empty(max(wsb, 1), dtype=torch.uint8, device=DEV)
    assert lib.rlctr_generate_preds_v10(L().ptr(dev(pctr)), L().ptr(dev(w)), L().ptr(dev(c)), L().ptr(dev(act.reshape(-1))),
                                        L().ptr(dev(lab.reshape(-1))), L().ptr(y), L().ptr(co), L().ptr(r), B, M, L().ptr(ws),
                                        wsb, st()) == 0
    return y.cpu().numpy(), r.cpu().numpy(), co.cpu().numpy()


@pytest.mark.parametrize("M", [3, 5, 6, 4])
def test_generate_preds_v10_golden(lib, golden_gp10, M):
    """src/all_main/hybrid_td3_main_per_v10.py:54-164 on the real reference's outputs: y to 1e-5, rewards and the returned
    c_actions (rank-indexed, :117) bit-exact."""
    g = lambda k: golden_gp10[f"gp10/M{M}/{k}"]
    y, r, co = _gp10(lib, g("pctr"), g("w"), g("c"), g("action"), g("label"))
    close(y, g("y").reshape(-1), rtol=1e-5, atol=1e-7)
    assert np.array_equal(r, g("reward").reshape(-1))
    assert np.array_equal(co, g("c_out"))


@pytest.mark.parametrize("B,M", [(1, 2), (255, 3), (5000, 8), (70001, 5), (300000, 6)])
def test_generate_preds_v10_random_vs_oracle(lib, B, M):
    """Ranks across many blocks (the scan over per-block counts), actions outside 1..M, every ensemble size."""
    rng = np.random.default_rng(B + M)
    pctr = rng.random((B, M)).astype(np.float32)
    w = O.softmax(rng.standard_normal((B, M)).astype(np.float32) * 2)
    c = np.tanh(rng.standard_normal((B, M))).astype(np.float32)
    lab = (rng.random(B) < 0.5).astype(np.int64)
    act = rng.integers(1, M + 1, size=B).astype(np.int64)
    act[::97] = 0
    act[5::1013] = M + 3
    y, r, co = _gp10(lib, pctr, w, c, act, lab)
    yo, ro, co_o, margin = O.generate_preds_v10(pctr, w, c, act, lab, return_margin=True)
    close(y, yo.reshape(-1), rtol=1e-5, atol=1e-7)
    assert np.array_equal(co, co_o)
    mism = r != ro.reshape(-1)
    assert not (mism & (margin > 2e-7)).any()          # two fp32 evaluations may disagree on a reward only at a tie


@pytest.mark.parametrize("variant", [0, 1])
def test_reinforce_head(lib, golden, variant):
    logits, acts = golden["pg/logits"], golden["pg/acts"].reshape(-1)
    B, A = logits.shape
    ws = torch.zeros(L().RLCTR_REDUCE_WS_BYTES, dtype=torch.uint8, device=DEV)
    for vt_key, loss_key, dl_key in (("pg/vt_norm", "pg/loss_literal", "pg/dlogits_literal"),
                                     ("pg/vt_raw", "pg/loss_literal_raw", "pg/dlogits_literal_raw")):
        vt = golden[vt_key].astype(np.float32)
        logp = torch.empty(B, device=DEV)
        loss = torch.empty(1, device=DEV)
        dl = torch.empty(B, A, device=DEV)
        assert lib.rlctr_reinforce_loss_bwd(L().ptr(dev(logits)), L().ptr(dev(acts)), L().ptr(dev(vt)), L().ptr(logp),
                                            L().ptr(loss), L().ptr(dl), L().ptr(ws), B, A, variant, st()) == 0
        close(logp, golden["pg/logp"], rtol=1e-5, atol=1e-7)                # policy log-probs: the 1e-5 bar
        lo, losso, dlo = O.reinforce_loss(logits, acts, vt, variant)
        close(logp, lo, rtol=1e-5, atol=1e-7)
        close(loss, losso, rtol=1e-4, atol=1e-5)
        close(dl, dlo, rtol=1e-4, atol=1e-7)
        if variant == 0:
            close(loss, golden[loss_key], rtol=1e-4, atol=2e-5)
            close(dl, golden[dl_key], rtol=1e-4, atol=1e-7)


# ------------------------------------------------------------------------------------------------
# K4 tcgen05 3xTF32 dense layers
# ------------------------------------------------------------------------------------------------
def linear_case(B, K, N, seed=0):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((B, K)).astype(np.float32)
    w = (rng.standard_normal((N, K)) / np.sqrt(K)).astype(np.float32)
    b = rng.standard_normal(N).astype(np.float32)
    return x, w, b


def padded(x, ld):
    """device copy of x [B, K] inside a [B, ld] buffer (pad columns hold NaN: nothing may read them)"""
    B, K = x.shape
    buf = torch.full((B, ld), float("nan"), device=DEV)
    buf[:, :K] = dev(x)
    return buf


# path: "tma" = 16-byte aligned pitch + workspace (TMA-fed kernel, csrc/mlp_tma.cu); "staged" = RLCTR_GEMM_TMA=0, dense x
# (software-staged kernel, csrc/mlp.cu: what any shape TMA cannot address falls back to).  K = 150 / 255 are not multiples of 4: "tma" pads the pitch.
# N = 75: a y pitch TMA cannot store to and a tile width (80) with a 16-column tail, so every column leaves by per-thread stores.
@pytest.mark.parametrize("B,K,N", [(1, 150, 300), (128, 32, 16), (1000, 150, 300), (777, 300, 200), (513, 200, 1),
                                   (1001, 203, 1), (1003, 256, 1), (6, 300, 1),
                                   (4096, 255, 1024), (300, 1024, 512), (65536, 150, 300), (999, 100, 75)])
@pytest.mark.parametrize("relu", [0, 1])
@pytest.mark.parametrize("path", ["tma", "staged"])
def test_linear_fwd_3xtf32(lib, B, K, N, relu, path, monkeypatch):
    monkeypatch.setenv("RLCTR_GEMM_TMA", "1" if path == "tma" else "0")
    x, w, b = linear_case(B, K, N, B + K + N)
    y = torch.empty(B, N, device=DEV)
    if path == "tma":
        ld = (K + 3) // 4 * 4
        xd = padded(x, ld)
        wsb = lib.rlctr_mlp_ws_bytes(B, K, N)
        ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
        rc = lib.rlctr_linear_fwd(L().ptr(xd), ld, L().ptr(dev(w)), L().ptr(dev(b)), L().ptr(y), B, K, N, relu, 0.0, None, L().ptr(ws), wsb, st())
    else:
        rc = lib.rlctr_linear_fwd(L().ptr(dev(x)), 0, L().ptr(dev(w)), L().ptr(dev(b)), L().ptr(y), B, K, N, relu, 0.0, None, None, 0, st())
    assert rc == 0
    ref = x.astype(np.float64) @ w.astype(np.float64).T + b
    if relu:
        ref = np.maximum(ref, 0)
    close(y, ref, rtol=1e-5)                 # fp32-grade: plain TF32 would be ~1e-3
    # and at least as close to the fp64 truth as fp32 SGEMM is, up to a small factor
    ref32 = x @ w.T + b
    if relu:
        ref32 = np.maximum(ref32, 0)
    err = np.abs(y.cpu().numpy() - ref).max()
    err32 = np.abs(ref32 - ref).max()
    assert err <= max(16 * err32, 2e-6 * np.abs(ref).max()), (err, err32)


@pytest.mark.parametrize("B,K,N", [(64, 150, 300), (1000, 150, 300), (777, 300, 200), (513, 200, 1), (65536, 300, 200),
                                   (65536, 150, 300), (4096, 255, 1024), (100, 64, 30)])
@pytest.mark.parametrize("relu", [0, 1])
@pytest.mark.parametrize("path", ["tma", "staged"])
def test_linear_bwd_3xtf32(lib, B, K, N, relu, path, monkeypatch):
    x, w, b = linear_case(B, K, N, B + K + N + 1)
    rng = np.random.default_rng(5)
    gy = rng.standard_normal((B, N)).astype(np.float32)
    y = np.maximum(x @ w.T + b, 0).astype(np.float32) if relu else None
    gyd = dev(gy)
    dx = torch.empty(B, K, device=DEV)
    dw = torch.empty(N, K, device=DEV)
    db = torch.empty(N, device=DEV)
    wsb = lib.rlctr_mlp_ws_bytes(B, K, N)
    ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
    monkeypatch.setenv("RLCTR_GEMM_TMA", "1" if path == "tma" else "0")
    if path == "tma":
        ld = (K + 3) // 4 * 4
        xd = padded(x, ld)
    else:
        ld, xd = K, dev(x)
    assert lib.rlctr_linear_bwd(L().ptr(xd), ld, L().ptr(dev(w)), L().ptr(dev(y)), L().ptr(gyd), L().ptr(dx), L().ptr(dw),
                                L().ptr(db), B, K, N, relu, 1.0, 1.0, L().ptr(ws), wsb, st()) == 0
    g64 = gy.astype(np.float64)
    if relu:
        g64 = g64 * (y > 0)
    close(dx, g64 @ w.astype(np.float64), rtol=1e-5)
    close(dw, g64.T @ x.astype(np.float64), rtol=1e-5)
    close(db, g64.sum(axis=0), rtol=1e-5)
    # deterministic split-K: bit-identical on a second run
    dw2 = torch.empty_like(dw)
    gyd2 = dev(gy)
    lib.rlctr_linear_bwd(L().ptr(xd), ld, L().ptr(dev(w)), L().ptr(dev(y)), L().ptr(gyd2), None, L().ptr(dw2), None, B, K, N,
                         relu, 1.0, 1.0, L().ptr(ws), wsb, st())
    assert torch.equal(dw, dw2)


@pytest.mark.parametrize("B,K,N", [(1, 7, 3), (64, 255, 300), (256, 259, 300), (300, 300, 3), (1000, 150, 300)])
@pytest.mark.parametrize("relu", [0, 1])
def test_linear_exact_fp32_path(lib, B, K, N, relu):
    """RLCTR_MLP_FP32: forward and backward on the CUDA cores, one FFMA per product -- fp32 SGEMM accuracy (1e-6 of the
    scale against float64, where the 3xTF32 kernels are allowed 1e-5), padded input rows, the masked dgrad and db included."""
    FP32 = 8
    x, w, b = linear_case(B, K, N, 21)
    ld = (K + 3) // 4 * 4 + 4
    xd = padded(x, ld)
    y = torch.empty(B, N, device=DEV)
    wsb = lib.rlctr_mlp_ws_bytes(B, K, N)
    ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
    assert lib.rlctr_linear_fwd(L().ptr(xd), ld, L().ptr(dev(w)), L().ptr(dev(b)), L().ptr(y), B, K, N, relu | FP32, 0.0, None,
                                L().ptr(ws), wsb, st()) == 0
    ref = x.astype(np.float64) @ w.astype(np.float64).T + b
    if relu:
        ref = np.maximum(ref, 0)
    close(y, ref, rtol=1e-6)
    gy = np.random.default_rng(5).standard_normal((B, N)).astype(np.float32)
    gyd = dev(gy)
    dx, dw, db = torch.empty(B, K, device=DEV), torch.empty(N, K, device=DEV), torch.empty(N, device=DEV)
    yh = y.cpu().numpy()
    assert lib.rlctr_linear_bwd(L().ptr(xd), ld, L().ptr(dev(w)), L().ptr(y), L().ptr(gyd), L().ptr(dx), L().ptr(dw), L().ptr(db),
                                B, K, N, relu | FP32 | 4, 1.0, 2.0, L().ptr(ws), wsb, st()) == 0
    g64 = gy.astype(np.float64) * ((yh > 0) if relu else 1.0)
    close(dx, (g64 @ w.astype(np.float64)) * np.where(x > 0, 2.0, 0.0), rtol=1e-6)        # RLCTR_MLP_DX_MASK: x is the mask source
    close(dw, g64.T @ x.astype(np.float64), rtol=1e-6)
    close(db, g64.sum(axis=0), rtol=1e-5)


@pytest.mark.parametrize("path", ["tma", "staged"])
@pytest.mark.parametrize("B,K,N", [(4096, 152, 300), (1000, 300, 200), (65536, 300, 200), (777, 100, 48), (40000, 36, 304)])
def test_linear_fused_dropout_and_masked_dgrad(lib, B, K, N, path, monkeypatch):
    """Forward: y = dropout(relu(x w^T + b)) with the counter-hash mask: kept elements equal relu(.)/(1-p), the kept fraction is
    1-p, the mask moves when the counter is advanced and repeats when it is not.  Backward of the layer above with
    RLCTR_MLP_DX_MASK: dx = (gy w) * (x > 0 ? s : 0) -- the mask-as-input reference (SURVEY N6)."""
    monkeypatch.setenv("RLCTR_GEMM_TMA", "1" if path == "tma" else "0")
    p = 0.2
    x, w, b = linear_case(B, K, N, 11)
    xd, wd, bd = dev(x), dev(w), dev(b)
    wsb = lib.rlctr_mlp_ws_bytes(B, K, N)
    ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
    rng = torch.tensor([1234567, 0], dtype=torch.int64, device=DEV)
    FL = 1 | 2
    y1, y2, y3 = (torch.empty(B, N, device=DEV) for _ in range(3))
    args = lambda y: (L().ptr(xd), K, L().ptr(wd), L().ptr(bd), L().ptr(y), B, K, N, FL, p, L().ptr(rng), L().ptr(ws), wsb, st())
    assert lib.rlctr_linear_fwd(*args(y1)) == 0
    assert lib.rlctr_linear_fwd(*args(y2)) == 0
    assert torch.equal(y1, y2)                                   # same (seed, counter) -> same mask
    assert lib.rlctr_rng_advance(L().ptr(rng), B * N, st()) == 0
    assert lib.rlctr_linear_fwd(*args(y3)) == 0
    ref = np.maximum(x.astype(np.float64) @ w.astype(np.float64).T + b, 0)
    y1n, y3n = y1.cpu().numpy(), y3.cpu().numpy()
    pos = ref > 1e-3 * np.abs(ref).max()
    kept = y1n[pos] != 0
    assert abs(kept.mean() - (1 - p)) < 0.01, kept.mean()
    assert abs((y3n[pos] != 0).mean() - (1 - p)) < 0.01
    assert ((y1n[pos] != 0) != (y3n[pos] != 0)).mean() > 0.2      # a different mask after the counter moved
    close(y1n[pos][kept], (ref[pos] / (1 - p))[kept], rtol=1e-5)
    pre = x.astype(np.float64) @ w.astype(np.float64).T + b
    assert (y1n[pre < -1e-5 * np.abs(pre).max()] == 0).all()     # clipped (beyond rounding of the pre-activation) -> 0
    # both kernels draw the same mask (the fused epilogue and the elementwise fallback share the hash)
    monkeypatch.setenv("RLCTR_GEMM_TMA", "0" if path == "tma" else "1")
    y4 = torch.empty(B, N, device=DEV)
    rng4 = torch.tensor([1234567, 0], dtype=torch.int64, device=DEV)
    assert lib.rlctr_linear_fwd(L().ptr(xd), K, L().ptr(wd), L().ptr(bd), L().ptr(y4), B, K, N, FL, p, L().ptr(rng4),
                                L().ptr(ws), wsb, st()) == 0
    assert torch.equal(y4 != 0, y1 != 0)
    monkeypatch.setenv("RLCTR_GEMM_TMA", "1" if path == "tma" else "0")
    # masked dgrad: x plays the role of the layer-below output (zeros where it was clipped / dropped)
    rs = np.random.default_rng(3)
    xm = np.where(rs.random((B, K)) < 0.4, 0.0, np.abs(x)).astype(np.float32)
    gy = rs.standard_normal((B, N)).astype(np.float32)
    dx = torch.empty(B, K, device=DEV)
    s = 1.0 / (1.0 - p)
    assert lib.rlctr_linear_bwd(L().ptr(dev(xm)), K, L().ptr(wd), None, L().ptr(dev(gy)), L().ptr(dx), None, None, B, K, N, 4,
                                1.0, s, L().ptr(ws), wsb, st()) == 0
    refdx = (gy.astype(np.float64) @ w.astype(np.float64)) * np.where(xm > 0, s, 0.0)
    close(dx, refdx, rtol=1e-5)
    assert (dx.cpu().numpy()[xm == 0] == 0).all()
    if path == "tma":                                    # the mask through TMA blocks == the mask read per thread, bit for bit
        # the same mask values at row pitch K + 1, which TMA cannot address: the kernel reads them per thread
        xmp = padded(xm, K + 1)
        dx2 = torch.empty(B, K, device=DEV)
        assert lib.rlctr_linear_bwd(L().ptr(xmp), K + 1, L().ptr(wd), None, L().ptr(dev(gy)), L().ptr(dx2), None, None, B, K, N, 4,
                                    1.0, s, L().ptr(ws), wsb, st()) == 0
        assert torch.equal(dx, dx2)


# ------------------------------------------------------------------------------------------------
# row sharding with G ranks emulated on ONE GPU: peers[] are G shard tensors in the same device memory
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_sort_and_peer_gather(lib, world):
    from rl_ctr_prediction_b200 import sharded
    N, B, F, rs, D = 5003, 300, 15, 16, 10
    rng = np.random.default_rng(world)
    full = rng.standard_normal((N, rs)).astype(np.float32)
    full[:, 11:] = 0
    n_max = sharded.shard_rows(N, world, 0)
    shards = []
    for r in range(world):
        sh = torch.zeros(n_max, rs, device=DEV)
        part = dev(full[r::world])
        sh[:part.shape[0]] = part
        shards.append(sh)
    ids = rng.integers(0, N, size=(world, B, F))
    ids[0, 0, 0] = N + 7
    # ---- rlctr_sort_ids_sharded against the host restatement, for every rank
    ids_all = torch.as_tensor(ids.reshape(-1)).to(DEV)
    all32 = ids_all.clamp(-1, N).to(torch.int32)
    n_all = all32.numel()
    for rank in range(world):
        srows = torch.empty(n_all, dtype=torch.int32, device=DEV)
        sslots = torch.empty(n_all, dtype=torch.int32, device=DEV)
        wsb = lib.rlctr_sort_ws_bytes(n_all, N)
        ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
        assert lib.rlctr_sort_ids_sharded(L().ptr(all32), n_all, world, rank, N, L().ptr(srows), L().ptr(sslots), L().ptr(ws),
                                          wsb, st()) == 0
        rows_h, pos_h = sharded.owned_sorted_view_host(ids_all.cpu(), world, rank, N)
        k = rows_h.numel()
        assert torch.equal(srows[:k].cpu().long(), rows_h) and torch.equal(sslots[:k].cpu().long(), pos_h)
        assert bool((srows[k:].cpu().long() == sharded.shard_rows(N, world, rank)).all())      # sentinel tail
    # ---- rlctr_embed_fwd through peers[]: same logits / sums / rows as the unsharded table
    x = torch.as_tensor(ids[1]).to(DEV)
    bias = dev(np.array([0.3], np.float32))
    outs = []
    for sharded_mode in (False, True):
        if sharded_mode:
            t = L().Table(shards[0].data_ptr(), N, rs, 0, 1, D, 0)
            t.world = world
            for r in range(world):
                t.peers[r] = shards[r].data_ptr()
        else:
            t = L().Table(L().ptr(dev(full)), N, rs, 0, 1, D, 0)
            keep = dev(full)
            t = L().Table(L().ptr(keep), N, rs, 0, 1, D, 0)
        logit = torch.empty(B, device=DEV)
        sums = torch.empty(B, rs, device=DEV)
        rows = torch.empty(B, F * D, device=DEV)
        assert lib.rlctr_embed_fwd(L().ptr(x), C.byref(t), L().ptr(bias), L().ptr(logit), None, 1, L().ptr(sums), L().ptr(rows), 0,
                                   B, F, 1, st()) == 0
        outs.append((logit.clone(), sums.clone(), rows.clone()))
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    # a world that is not a power of two, or a missing peer, is refused
    t.world = 3
    assert lib.rlctr_embed_fwd(L().ptr(x), C.byref(t), L().ptr(bias), L().ptr(logit), None, 1, None, None, 0, B, F, 1, st()) == -2
    t.world = world
    t.peers[world - 1] = None
    assert lib.rlctr_embed_fwd(L().ptr(x), C.byref(t), L().ptr(bias), L().ptr(logit), None, 1, None, None, 0, B, F, 1, st()) == -2


@pytest.mark.parametrize("world", [2, 4, 8])
def test_owner_routing_equals_gather_and_sort(lib, world):
    """rlctr_route_ids (every source writes the (local row, global slot) pairs a peer owns into that peer's receive buffer)
    + rlctr_sort_routed == the all-gather + rlctr_sort_ids_sharded view == the host restatement, for every owner; G ranks
    emulated on one GPU (the receive buffers of all owners live in the same memory).  A bucket beyond the capacity raises
    the overflow flag."""
    from rl_ctr_prediction_b200 import sharded
    N, B, F = 5003, 300, 15
    n = B * F
    rng = np.random.default_rng(100 + world)
    ids = rng.integers(0, N, size=(world, B, F))
    ids[0, 0, 0] = N + 7                                  # out of range: routed nowhere
    ids[1, 2, :] = ids[1, 3, :]                           # duplicates
    cap = sharded.route_capacity(n, world)
    keys = [torch.full((world * cap,), -1, dtype=torch.int32, device=DEV) for _ in range(world)]
    vals = [torch.zeros(world * cap, dtype=torch.int32, device=DEV) for _ in range(world)]
    kp = (C.c_void_p * 8)(*[k.data_ptr() for k in keys])
    vp = (C.c_void_p * 8)(*[v.data_ptr() for v in vals])
    flag = torch.zeros(1, dtype=torch.int32, device=DEV)
    wsb = lib.rlctr_route_ws_bytes(n, world)
    ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
    for src in range(world):                              # every source rank routes its batch
        x = dev(ids[src].reshape(-1))
        assert lib.rlctr_route_ids(L().ptr(x), n, world, src, N, cap, kp, vp, L().ptr(flag), L().ptr(ws), wsb, st()) == 0
    assert int(flag.item()) == 0
    ids_all = torch.as_tensor(ids.reshape(-1))
    for owner in range(world):
        n_in = world * cap
        n_local = sharded.shard_rows(N, world, owner)
        srows = torch.empty(n_in, dtype=torch.int32, device=DEV)
        sslots = torch.empty(n_in, dtype=torch.int32, device=DEV)
        wsb2 = lib.rlctr_sort_ws_bytes(n_in, n_local)
        ws2 = torch.empty(wsb2, dtype=torch.uint8, device=DEV)
        assert lib.rlctr_sort_routed(L().ptr(keys[owner]), L().ptr(vals[owner]), n_in, n_local, L().ptr(srows), L().ptr(sslots),
                                     L().ptr(ws2), wsb2, st()) == 0
        rows_h, pos_h = sharded.owned_sorted_view_host(ids_all, world, owner, N)
        k = rows_h.numel()
        assert torch.equal(srows[:k].cpu().long(), rows_h) and torch.equal(sslots[:k].cpu().long(), pos_h)
        assert bool((srows[k:].cpu() == -1).all())        # sentinel tail (0xffffffff >= any row count)
    # overflow: a capacity below the largest bucket
    small = max(n // world // 4, 1)
    k2 = [torch.empty(world * small, dtype=torch.int32, device=DEV) for _ in range(world)]
    v2 = [torch.empty(world * small, dtype=torch.int32, device=DEV) for _ in range(world)]
    kp2 = (C.c_void_p * 8)(*[k.data_ptr() for k in k2])
    vp2 = (C.c_void_p * 8)(*[v.data_ptr() for v in v2])
    assert lib.rlctr_route_ids(L().ptr(dev(ids[0].reshape(-1))), n, world, 0, N, small, kp2, vp2, L().ptr(flag), L().ptr(ws), wsb,
                               st()) == 0
    assert int(flag.item()) != 0


@pytest.mark.parametrize("dz_in_sums", [0, 1])
@pytest.mark.parametrize("world", [2, 4])
def test_sharded_owner_update_equals_single_table(lib, world, dz_in_sums):
    """G ranks' FM steps emulated on one GPU: each owner runs rlctr_rows_adam on its shard with the sorted owned view
    and PULLS dlogit / sums / extra from the G source buffers (peer_* pointers); the union of the shards equals one
    rlctr_rows_adam over the whole table with the concatenated batch -- bit for bit."""
    from rl_ctr_prediction_b200 import sharded
    from rl_ctr_prediction_b200.tables import AdamSchedule
    N, B, F, rs, D = 3001, 200, 15, 16, 10
    rng = np.random.default_rng(5 + world)
    full = rng.standard_normal((N, rs)).astype(np.float32) * 0.1
    full[:, 11:] = 0
    ids = rng.integers(0, N, size=(world, B, F))
    dl = [rng.standard_normal(B).astype(np.float32) * 0.01 for _ in range(world)]
    sm = [rng.standard_normal((B, rs)).astype(np.float32) for _ in range(world)]
    ex = [rng.standard_normal((B, F * D)).astype(np.float32) * 0.01 for _ in range(world)]
    sched = AdamSchedule(1e-3, (0.9, 0.999), DEV)

    def adam_struct(tab):
        m, v = torch.zeros_like(tab), torch.zeros_like(tab)
        step = torch.zeros(1, dtype=torch.int32, device=DEV)
        a = L().Adam(m.data_ptr(), v.data_ptr(), None, L().ptr(sched.tensor), L().ptr(step), sched.length, -1, 0.9, 0.999, 1e-8, 1e-5)
        return a, (m, v, step)

    # ---- reference: one table, concatenated batch
    tab = dev(full)
    x_all = torch.as_tensor(ids.reshape(-1, F)).to(DEV)
    sid = torch.empty(x_all.numel(), dtype=torch.int32, device=DEV)
    ssl = torch.empty_like(sid)
    wsb = lib.rlctr_sort_ws_bytes(x_all.numel(), N)
    ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
    assert lib.rlctr_sort_ids(L().ptr(x_all), x_all.numel(), N, L().ptr(sid), L().ptr(ssl), L().ptr(ws), wsb, st()) == 0
    dl_all, sm_all, ex_all = dev(np.concatenate(dl)), dev(np.concatenate(sm)), dev(np.concatenate(ex))
    g = L().RowGrad(None, L().ptr(dl_all), L().ptr(sm_all), L().ptr(ex_all), F, 0)
    t = L().Table(L().ptr(tab), N, rs, 0, 1, D, 0)
    a, keep = adam_struct(tab)
    rwb = lib.rlctr_rows_ws_bytes(x_all.numel())
    rws = torch.empty(rwb, dtype=torch.uint8, device=DEV)
    assert lib.rlctr_rows_adam(L().ptr(sid), L().ptr(ssl), x_all.numel(), C.byref(g), C.byref(t), C.byref(a), L().ptr(rws), rwb, st()) == 0
    # ---- sharded: per owner
    if dz_in_sums:                     # RLCTR_DZ_IN_SUMS: dlogit rides in the last (padding) column of the sums row
        for r in range(world):
            sm[r] = sm[r].copy()
            sm[r][:, rs - 1] = dl[r]
    dls, sms, exs = [dev(d) for d in dl], [dev(s) for s in sm], [dev(e) for e in ex]
    all32 = x_all.reshape(-1).to(torch.int32)
    n_all = all32.numel()
    for rank in range(world):
        n_local = sharded.shard_rows(N, world, rank)
        shard = dev(full[rank::world])
        srows = torch.empty(n_all, dtype=torch.int32, device=DEV)
        sslots = torch.empty(n_all, dtype=torch.int32, device=DEV)
        assert lib.rlctr_sort_ids_sharded(L().ptr(all32), n_all, world, rank, N, L().ptr(srows), L().ptr(sslots), L().ptr(ws), wsb,
                                          st()) == 0
        gs = L().RowGrad(None, None, None, None, F, 2 if dz_in_sums else 0)
        gs.world, gs.n_per_rank = world, B * F
        for r in range(world):
            gs.peer_dlogit[r], gs.peer_sums[r], gs.peer_extra[r] = dls[r].data_ptr(), sms[r].data_ptr(), exs[r].data_ptr()
        ts = L().Table(L().ptr(shard), n_local, rs, 0, 1, D, 0)
        as_, keep2 = adam_struct(shard)
        assert lib.rlctr_rows_adam(L().ptr(srows), L().ptr(sslots), n_all, C.byref(gs), C.byref(ts), C.byref(as_), L().ptr(rws), rwb,
                                   st()) == 0
        assert torch.equal(shard, tab[rank::world]), rank
        assert torch.equal(keep2[0], keep[0][rank::world]) and torch.equal(keep2[1], keep[1][rank::world])


# ------------------------------------------------------------------------------------------------
# device AUC / log-loss (SURVEY 8f.3) against sklearn
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["random", "ties", "saturated", "tiny", "large"])
def test_auc_logloss_matches_sklearn(lib, case):
    from sklearn.metrics import log_loss, roc_auc_score
    from rl_ctr_prediction_b200 import metrics
    rng = np.random.default_rng(7)
    n = {"random": 10007, "ties": 5000, "saturated": 4096, "tiny": 2, "large": 1 << 20}[case]
    y = (rng.random(n) < 0.2).astype(np.int64)
    if case == "tiny":
        y = np.array([0, 1], np.int64)
    p = rng.random(n).astype(np.float32)
    p = np.clip(0.6 * p + 0.4 * y * rng.random(n).astype(np.float32), 1e-6, 1 - 1e-6).astype(np.float32)
    if case == "ties":
        p = (np.round(p * 8) / 8).astype(np.float32).clip(0.0625, 0.9375)          # 8 distinct scores
    if case == "saturated":
        p[: n // 2] = np.where(rng.random(n // 2) < 0.5, 0.0, 1.0).astype(np.float32)   # exact 0 / 1 like N(0,1) init (SURVEY N2)
    out = metrics.auc_logloss(dev(p), torch.as_tensor(y).to(DEV)).cpu().numpy()
    assert abs(out[0] - roc_auc_score(y, p)) < 2e-6
    pc = p.astype(np.float64)
    ll = np.mean(-(y * np.maximum(np.log(pc), -100)) - (1 - y) * np.maximum(np.log1p(-pc), -100)) if case != "saturated" else None
    if ll is not None:
        assert abs(out[1] - ll) < 1e-5 * max(1.0, abs(ll))
    # float labels, and run-to-run determinism
    out2 = metrics.auc_logloss(dev(p), dev(y.astype(np.float32))).cpu().numpy()
    assert np.array_equal(out, out2)
    # one class only: AUC undefined (sklearn raises; here NaN)
    assert np.isnan(metrics.auc_logloss(dev(p), torch.zeros(n, dtype=torch.int64, device=DEV)).cpu().numpy()[0])


@pytest.mark.parametrize("B,N,relu", [(256, 300, True), (16, 5, True), (1000, 33, False), (4096, 128, True)])
def test_bn_relu_matches_torch(B, N, relu):
    """rlctr_bn_relu_fwd / _bwd (training-mode BatchNorm1d [+ ReLU], the policy nets' hidden layers in their learn steps,
    DDQN_model.py:32-46) against torch's own BatchNorm1d + ReLU in float64: outputs, input / gamma / beta gradients, running
    statistics (momentum, unbiased variance) and num_batches_tracked."""
    from rl_ctr_prediction_b200 import mlp
    torch.manual_seed(B + N)
    bn = torch.nn.BatchNorm1d(N).to(DEV).train()
    with torch.no_grad():
        bn.weight.uniform_(0.5, 1.5)
        bn.bias.normal_()
        bn.running_mean.normal_()
        bn.running_var.uniform_(0.5, 2.0)
    ref = torch.nn.BatchNorm1d(N).to(DEV).double().train()
    ref.load_state_dict({k: v.double() if v.is_floating_point() else v for k, v in bn.state_dict().items()})
    base = torch.randn(B, N + 3, device=DEV) * 2.0 + 0.7
    x = base[:, :N].detach().requires_grad_(True)                        # a pitched view, like the GEMM outputs the kernel is fed
    xr = base[:, :N].double().detach().requires_grad_(True)
    gy = torch.randn(B, N, device=DEV)
    y = mlp.bn_relu(bn, x, relu)
    yr = ref(xr)
    close(y, torch.relu(yr) if relu else yr, rtol=1e-5)
    # the backward takes the ReLU mask of the kernel's own output (mask as input): an activation within rounding of zero may fall
    # on either side in fp32 / fp64, and one flipped element shifts the column sums -- and with them the whole column of dx
    yr = yr * (y > 0).double() if relu else yr
    y.backward(gy)
    yr.backward(gy.double())
    close(x.grad, xr.grad, rtol=1e-5)
    close(bn.weight.grad, ref.weight.grad, rtol=1e-5)
    close(bn.bias.grad, ref.bias.grad, rtol=1e-5)
    close(bn.running_mean, ref.running_mean, rtol=1e-5)
    close(bn.running_var, ref.running_var, rtol=1e-5)
    assert int(bn.num_batches_tracked) == int(ref.num_batches_tracked) == 1
    # the Tower routes a training-mode Linear -> BatchNorm1d -> ReLU stack through it: same numbers as the same stack with torch's
    # own BatchNorm1d / ReLU modules between the same GEMMs (fusion switched off)
    import copy
    from rl_ctr_prediction_b200 import DDQN_model
    torch.manual_seed(1)
    net = DDQN_model.bn_mlp(N, 3, hidden=(64, 32), device=DEV).train()
    twin = copy.deepcopy(net)
    inp = torch.randn(B, N, device=DEV)
    out = net(inp)
    out.sum().backward()
    saved, mlp.BN_FUSED_MAX_BATCH = mlp.BN_FUSED_MAX_BATCH, 0
    try:
        out_ref = twin(inp)
        out_ref.sum().backward()
    finally:
        mlp.BN_FUSED_MAX_BATCH = saved
    close(out, out_ref, rtol=2e-5)
    for (k, p), (_, q) in zip(net.named_parameters(), twin.named_parameters()):
        # every one of these gradients is a sum over the B samples of O(1) terms that largely cancel (the loss is out.sum()), so
        # two correct fp32 evaluations differ by ~1e-7 * B in absolute terms; the biases in front of a BatchNorm have an exactly
        # zero gradient (the batch mean is subtracted again) and carry nothing but that noise
        if k in ("0.bias", "3.bias"):
            assert float(p.grad.abs().max()) <= 5e-6 * B and float(q.grad.abs().max()) <= 5e-6 * B, k
            continue
        close(p.grad, q.grad, rtol=5e-5, atol=max(5e-5 * float(q.grad.abs().max()), 1e-6 * B)), k
    for (k, u), (_, v) in zip(net.named_buffers(), twin.named_buffers()):
        close(u.float(), v.float(), rtol=1e-5), k


def _plain_linear(m):
    lin = torch.nn.Linear(m.in_features, m.out_features, device=m.weight.device)
    lin.load_state_dict(m.state_dict())
    return lin
