"""Field-count limits without a GPU: InnerPNN's pair dots and FFM serve 2 <= F <= 64 and refuse F = 65 with RLCTR_EUNSUPPORTED
before any CUDA call, the error names the new limits, the limits that stay (AFM F <= 23, DCN F*D <= 512, FFM rows of 512 floats)
keep their messages, and the pair-index formula of the kernels' tables needs 16-bit entries from F = 24 on."""
import ctypes as C

import pytest
import torch

from rl_ctr_prediction_b200 import _lib

EINVAL, EUNSUPPORTED = -1, -2
_FAKE = 1 << 20                     # 16-byte aligned stand-in address: every call below returns before reading through it


def _ffm_table(F, D, n_rows=1000):
    rs = (F * D + 1 + 3) // 4 * 4
    return _lib.Table(_FAKE, n_rows, rs, F * D, 0, F * D, 0)


def test_pairdots_past_64_fields_are_refused():
    lib = _lib.load()
    for F, D in ((65, 1), (65, 8), (100, 4)):
        fd, P = F * D, F * (F - 1) // 2
        assert lib.rlctr_pairdots_fwd(_FAKE, fd, _FAKE, fd + P, 64, F, D, 0, None) == EUNSUPPORTED
        assert lib.rlctr_pairdots_bwd(_FAKE, fd, _FAKE, fd + P, _FAKE, fd, 64, F, D, 1, None) == EUNSUPPORTED
    # bad arguments at the new field counts are still EINVAL
    F, D = 64, 8
    fd, P = F * D, F * (F - 1) // 2
    assert lib.rlctr_pairdots_fwd(_FAKE, fd, _FAKE, fd + P - 1, 64, F, D, 0, None) == EINVAL          # ld_out < F*D + P
    assert lib.rlctr_pairdots_bwd(_FAKE, fd - 1, _FAKE, fd + P, _FAKE, fd, 64, F, D, 0, None) == EINVAL
    assert lib.rlctr_pairdots_fwd(_FAKE, fd, _FAKE, fd + P, 64, 1, D, 0, None) == EINVAL                # F = 1
    # the byte-table path keeps its 48 KB cap: F = 23 at a D whose stage needs more is still refused
    F, D = 23, 200
    fd, P = F * D, F * (F - 1) // 2
    assert lib.rlctr_pairdots_fwd(_FAKE, fd, _FAKE, fd + P, 64, F, D, 0, None) == EUNSUPPORTED


def test_ffm_past_64_fields_and_512_float_rows_are_refused():
    lib = _lib.load()
    for F, D in ((65, 1), (65, 7), (128, 2)):
        t = _ffm_table(F, D)
        assert lib.rlctr_ffm_fwd(_FAKE, C.byref(t), None, _FAKE, None, 1, _FAKE, 64, F, D, None) == EUNSUPPORTED
    # one sample's rows past 227 KB of shared memory (F = 64 at 772-float rows)
    t = _ffm_table(64, 12)
    assert lib.rlctr_ffm_fwd(_FAKE, C.byref(t), None, _FAKE, None, 1, _FAKE, 64, 64, 12, None) == EUNSUPPORTED
    t = _ffm_table(64, 7)
    t.dim = 64 * 7 + 1                                                                    # dim != F * D
    assert lib.rlctr_ffm_fwd(_FAKE, C.byref(t), None, _FAKE, None, 1, _FAKE, 64, 64, 7, None) == EINVAL
    # the update keeps FFM rows at 512 floats: F = 64, D = 8 is 513 -> 516 floats, F = 39, D = 14 is 547 -> 548
    a = _lib.Adam(_FAKE, _FAKE, None, _FAKE, _FAKE, 1, -1, 0.9, 0.999, 1e-8, 0.0, None)
    for F, D in ((64, 8), (39, 14)):
        t = _ffm_table(F, D)
        g = _lib.RowGrad(_FAKE, _FAKE, None, None, F, _lib.RLCTR_STAGED_PARTNER)
        assert lib.rlctr_rows_adam(_FAKE, _FAKE, 64, C.byref(g), C.byref(t), C.byref(a), _FAKE, 1 << 20, None) == EUNSUPPORTED


def test_errors_name_the_field_limits():
    lib = _lib.load()
    F, D = 65, 4
    fd, P = F * D, F * (F - 1) // 2
    with pytest.raises(_lib.RlctrError, match=r"F <= 64"):
        _lib.call("rlctr_pairdots_fwd", lib.rlctr_pairdots_fwd, _FAKE, fd, _FAKE, fd + P, 64, F, D, 0, None)
    with pytest.raises(_lib.RlctrError, match=r"F <= 64"):
        _lib.call("rlctr_pairdots_bwd", lib.rlctr_pairdots_bwd, _FAKE, fd, _FAKE, fd + P, _FAKE, fd, 64, F, D, 0, None)
    t = _ffm_table(F, D)
    with pytest.raises(_lib.RlctrError, match=r"F <= 64"):
        _lib.call("rlctr_ffm_fwd", lib.rlctr_ffm_fwd, _FAKE, C.byref(t), None, _FAKE, None, 1, _FAKE, 64, F, D, None)
    assert "48 KB" in _lib.SHAPE_LIMITS["rlctr_group_fwd"] and "128 floats" in _lib.SHAPE_LIMITS["rlctr_group_fwd"]


def test_limits_that_stay_keep_their_messages():
    lib = _lib.load()
    assert _lib.SHAPE_LIMITS["rlctr_afm_fwd"] == "AFM: D <= 32, F <= 23"
    assert _lib.SHAPE_LIMITS["rlctr_afm_bwd"] == "AFM: D <= 32, F <= 23"
    assert _lib.SHAPE_LIMITS["rlctr_cross_fwd"] == "DCN: F*D <= 512, at most 8 cross layers"
    assert _lib.SHAPE_LIMITS["rlctr_cross_bwd"] == "DCN: F*D <= 512, at most 6 cross layers"
    assert _lib.SHAPE_LIMITS["rlctr_embed_fwd"] == ("fused rows of at most 36 floats (D <= 32 with a first-order column, "
                                                    "36 without)")
    for F in (24, 39, 64):                                                                 # AFM stays at F <= 23
        with pytest.raises(_lib.RlctrError, match=r"D <= 32, F <= 23"):
            _lib.call("rlctr_afm_fwd", lib.rlctr_afm_fwd, _FAKE, F * 8, _FAKE, _FAKE, 64, F, 8, 0.0, None, None, None)
    fd = 39 * 14                                                                           # DCN at F = 39 past D = 13
    with pytest.raises(_lib.RlctrError, match=r"F\*D <= 512"):
        _lib.call("rlctr_cross_fwd", lib.rlctr_cross_fwd, _FAKE, fd, _FAKE, _FAKE, 5, _FAKE, fd, _FAKE, 64, fd, None)


def _pair(i, j, F):
    """Mirror of the kernels' pair index of (i, j), i < j (csrc/embed.cu pair_tables, csrc/ffm.cu)."""
    return i * F - i * (i + 1) // 2 + j - i - 1


def test_pair_index_formula_matches_triu_order():
    for F in range(2, 65):
        iu = torch.triu_indices(F, F, offset=1)
        got = [_pair(int(i), int(j), F) for i, j in zip(iu[0], iu[1])]
        assert got == list(range(F * (F - 1) // 2)), F
        top = _pair(F - 2, F - 1, F)
        assert top == F * (F - 1) // 2 - 1
        assert (top > 255) == (F >= 24), F                # byte pair indices hold F <= 23 only
        assert top < 1 << 16                              # 16-bit entries hold every F up to 64 (2015 at F = 64)
    assert _pair(62, 63, 64) == 2015
