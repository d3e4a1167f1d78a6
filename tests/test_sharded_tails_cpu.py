"""Row-sharded tail models without a GPU: the multi-source routed push checks its arguments before any CUDA call, and ShardedCTR /
ShardedGroup refuse what they cannot shard before they touch a device."""
import ctypes as C

import pytest

from rl_ctr_prediction_b200 import _lib, sharded

# stand-in addresses: every call below fails its argument check and returns before anything is read through them
_FAKE = 1 << 20


def _call(lib, route_ws=_FAKE, n=40, world=2, rank=0, cap=256, srcs=(_FAKE,), widths=(10,), n_src=None, peers=(_FAKE, _FAKE)):
    s = (C.c_void_p * max(len(srcs), 1))(*srcs) if srcs is not None else None
    w = (C.c_int32 * max(len(widths), 1))(*widths) if widths is not None else None
    p = (C.c_void_p * 8)(*peers) if peers is not None else None
    return lib.rlctr_push_rows_routed_multi(route_ws, n, world, rank, cap, s, w, len(srcs or ()) if n_src is None else n_src, p, None)


def test_push_rows_routed_multi_rejects_bad_arguments():
    lib = _lib.load()
    EINVAL = -1
    assert _call(lib, route_ws=None) == EINVAL
    assert _call(lib, srcs=None) == EINVAL
    assert _call(lib, widths=None) == EINVAL
    assert _call(lib, srcs=(_FAKE, 0), widths=(10, 10)) == EINVAL              # a NULL source
    assert _call(lib, widths=(9,)) == EINVAL                                    # odd width: 8-byte pieces
    assert _call(lib, widths=(0,)) == EINVAL
    assert _call(lib, n_src=0) == EINVAL
    assert _call(lib, srcs=(_FAKE,) * 5, widths=(10,) * 5) == EINVAL           # more than RLCTR_GROUP_MAX sources
    assert _call(lib, rank=2) == EINVAL
    assert _call(lib, cap=0) == EINVAL
    assert _call(lib, n=-1) == EINVAL
    assert _call(lib, peers=None) == EINVAL
    assert _call(lib, peers=(_FAKE, 0)) == EINVAL                               # a NULL receive buffer
    for world in (1, 3, 16):
        assert _call(lib, world=world, peers=(_FAKE,) * 8) not in (0,)
    assert _call(lib, srcs=(_FAKE + 4,)) != 0                                   # misaligned source rows
    # the one-source call keeps its contract
    assert lib.rlctr_push_rows_routed(None, 4, 2, 0, 8, None, 10, None, None) == EINVAL


def test_sharded_models_refuse_what_they_cannot_shard():
    with pytest.raises(_lib.RlctrError):
        sharded.ShardedGroup(("FM", "FFM"), 1000, 15, 10, device="cpu")
    with pytest.raises(_lib.RlctrError):
        sharded.ShardedGroup(("FM", "Bogus"), 1000, 15, 10, device="cpu")
    with pytest.raises(_lib.RlctrError):
        sharded.ShardedGroup(("LR",) * 5, 1000, 15, 10, device="cpu")
    with pytest.raises(_lib.RlctrError):                                        # three vector members: wider than one line
        sharded.ShardedGroup(("FM", "FNN", "DeepFM"), 1000, 15, 10, device="cpu")
    with pytest.raises(_lib.RlctrError):
        sharded.ShardedCTR("Bogus", 1000, 15, 10, device="cpu")


def test_tail_kind_names():
    assert set(sharded.TAIL_KINDS) == {"WideAndDeep", "FNN", "InnerPNN", "OuterPNN", "DCN", "AFM"}
    from rl_ctr_prediction_b200 import colocated
    assert {c.__name__ for c in colocated.MEMBER_KINDS} == set(sharded.TAIL_KINDS) | {"LR", "FM", "DeepFM"}
