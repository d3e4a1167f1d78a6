"""Wide co-located records without a GPU: colocated._layout(max_lines=...) places the columns and refuses what does not fit, with
messages that say which limit was hit; ShardedGroup refuses before it touches a device; the C entry points refuse wide tables they
cannot serve before any CUDA call."""
import ctypes as C

import pytest

from rl_ctr_prediction_b200 import _lib, colocated, sharded
from rl_ctr_prediction_b200.tables import Geometry, round4

N = 1000


class M:
    def __init__(self, g):
        self._geom = g


def lr():
    return M(Geometry.lr(N))


def fm(d):
    return M(Geometry.fm(N, d))


def fnn(d):
    return M(Geometry.fm(N, d, with_linear=False))


@pytest.mark.parametrize("max_lines", [2, 3, 4])
@pytest.mark.parametrize("d", [1, 10, 15, 16, 20, 31, 32])
def test_layout_keeps_standalone_alignment(max_lines, d):
    """FM + FNN + LR: vector members from chunk boundaries with their stand-alone columns, LR in a padding column or a chunk of its
    own, the stamp in the last active chunk; four lines hold every latent size."""
    members = [fm(d), fnn(d), lr()]
    try:
        cols, used = colocated._layout(members, max_lines)
    except _lib.RlctrError as e:
        assert max_lines < 4 and "max_lines" in str(e)
        return
    (lf, ef, df), (ln, en, dn), (ll, _, _) = cols
    assert lf % 4 == 0 and ef == lf + 1 and df == d                       # FM: [w, v..] from a chunk boundary, as stand-alone
    assert ln == -1 and en == round4(d + 1) and dn == d                   # FNN: [v..] from where FM's row ends
    taken = {lf, *range(ef, ef + d), *range(en, en + d), ll}
    assert len(taken) == 2 * d + 2                                        # no column shared
    top = max(taken) + 1
    assert used == (top + 1 if top % 4 == 0 else top)                     # the stamp: a free column of the last active chunk
    rs = round4(used + 1)
    assert rs <= 32 * max_lines
    rec = colocated._record(N, used)
    assert rec.stamp_col == used and rec.row_pitch % 32 == 0 and rec.row_pitch >= 3 * rs
    if rs <= 32:
        assert (rec.row_pitch, rec.block_floats) == (96, 32)
    else:
        assert (rec.block_floats, rec.row_pitch) == (rs, (3 * rs + 31) // 32 * 32)


def test_member_views_of_a_wide_record():
    """Each member of a wide record sees its stand-alone row: from its first chunk, its own row_stride, the joint pitch."""
    members = [lr(), fm(20), fm(20)]
    cols, used = colocated._layout(members, 2)
    rec = colocated._record(N, used)
    assert colocated._wide(members, used)
    views = [colocated._member_view(m, rec, c, True) for m, c in zip(members, cols)]
    assert (views[0].row_stride, views[0].lin_col, views[0].offset) == (1, 0, cols[0][0])
    for m, v, (lin, emb, dim) in zip(members[1:], views[1:], cols[1:]):
        g = m._geom
        assert (v.row_stride, v.lin_col, v.emb_col, v.dim) == (g.row_stride, g.lin_col, g.emb_col, g.dim)
        assert v.offset + v.lin_col == lin and v.offset + v.emb_col == emb and v.row_pitch == rec.row_pitch


def test_layout_refusals_name_the_limit():
    with pytest.raises(_lib.RlctrError, match="max_lines=2") as e:
        colocated._layout([fm(10), fm(10), fm(10)])                       # fits two lines
    assert "max_lines" in str(e.value) and "32 floats" in str(e.value)
    with pytest.raises(_lib.RlctrError) as e:
        colocated._layout([fm(16)])                                       # a 20-float row: not beside one-line members
    assert "max_lines" in str(e.value) and "32 floats" in str(e.value) and "FFM" not in str(e.value)
    with pytest.raises(_lib.RlctrError, match="4 lines"):
        colocated._layout([fm(32)] * 4, 4)                                # 4 x 36 floats: wider than four lines
    for ml in (1, 2, 4):
        with pytest.raises(_lib.RlctrError, match="FFM"):
            colocated._layout([M(Geometry.ffm(N, 15, 10))], ml)
        with pytest.raises(_lib.RlctrError, match="FFM"):
            colocated._layout([fm(4), M(Geometry.ffm(N, 2, 2))], ml)     # a narrow FFM row is still FFM
    for bad in (0, 5):
        with pytest.raises(ValueError):
            colocated._layout([fm(10)], bad)
    colocated._layout([fm(16)], 2)
    colocated._layout([fm(32), fm(32), lr()], 3)


def test_sharded_group_refusals():
    with pytest.raises(_lib.RlctrError, match="max_lines"):              # rs 32: the one-line exchange row holds 28
        sharded.ShardedGroup(("LR", "FM", "DeepFM"), N, 15, 12, device="cpu")
    with pytest.raises(_lib.RlctrError, match="FFM"):
        sharded.ShardedGroup(("FM", "FFM"), N, 15, 10, device="cpu", max_lines=4)
    with pytest.raises(_lib.RlctrError, match="4 lines"):
        sharded.ShardedGroup(("FM", "DeepFM", "FNN", "WideAndDeep"), N, 15, 32, device="cpu", max_lines=4)
    with pytest.raises(ValueError):
        sharded.ShardedGroup(("FM", "DeepFM"), N, 15, 10, device="cpu", max_lines=5)


_FAKE = 1 << 20        # stand-in device address: every call below returns before anything is read through it


def _table(rs, used, pitch):
    return _lib.Table(_FAKE, 100, rs, -1, 0, used, pitch)


def _member(lin, emb, dim, fm_term=True):
    m = _lib.Member()
    m.lin_col, m.emb_col, m.dim, m.flags = lin, emb, dim, _lib.RLCTR_FM_TERM if fm_term else 0
    return m


def test_entry_points_refuse_wide_tables_before_any_cuda_call():
    lib = _lib.load()
    EINVAL, EUNSUP = -1, -2
    ids = _FAKE
    arr = (_lib.Member * 1)(_member(0, 1, 32))
    # a joint row wider than four lines
    t = _table(132, 130, 132 * 3)
    assert lib.rlctr_group_fwd(ids, C.byref(t), arr, 1, None, 0, 8, 15, None) == EUNSUP
    a = _lib.Adam(_FAKE, _FAKE, None, _FAKE, _FAKE, 100, 130, 0.9, 0.999, 1e-8, 0.0, None)
    assert lib.rlctr_group_rows_adam(ids, ids, 8, C.byref(t), C.byref(a), arr, 1, _FAKE, 0, 15, 1, None, _FAKE, 1 << 20,
                                     None) == EUNSUP
    # a member whose stand-alone row would be wider than 36 floats
    t = _table(64, 41, 224)
    arr2 = (_lib.Member * 1)(_member(0, 1, 40))
    assert lib.rlctr_group_fwd(ids, C.byref(t), arr2, 1, None, 0, 8, 15, None) == EUNSUP
    # member columns outside the row, bad counts
    t = _table(72, 69, 224)
    assert lib.rlctr_group_fwd(ids, C.byref(t), (_lib.Member * 1)(_member(0, 60, 32)), 1, None, 0, 8, 15, None) == EINVAL
    assert lib.rlctr_group_fwd(ids, C.byref(t), arr, 5, None, 0, 8, 15, None) == EINVAL
    assert lib.rlctr_group_fwd(ids, C.byref(t), arr, 1, None, 70, 8, 15, None) == EINVAL     # sums pitch < row_stride
    # two FM-term members in one chunk
    two = (_lib.Member * 2)(_member(0, 1, 16), _member(-1, 17, 16))
    assert lib.rlctr_group_fwd(ids, C.byref(t), two, 2, None, 0, 8, 15, None) == EUNSUP
    # catch-up / flush of an in-record-stamp record wider than four lines
    t = _table(132, 130, 132 * 3)
    assert lib.rlctr_rows_catchup(ids, 8, C.byref(t), C.byref(a), None) == EUNSUP
    assert lib.rlctr_adam_flush(C.byref(t), C.byref(a), 0, 100, None) == EUNSUP
    # the batch-order catch-up serves records of 5..8 chunks only
    t = _table(72, 69, 224)
    a.stamp_col = 69
    assert lib.rlctr_rows_catchup_ids(ids, 8, C.byref(t), C.byref(a), _FAKE, lib.rlctr_rows_claim_bytes(100), None) == EUNSUP


def test_shape_limits_name_the_group_limit():
    for name in ("rlctr_group_fwd", "rlctr_group_rows_adam"):
        assert "128 floats" in _lib.SHAPE_LIMITS[name]
