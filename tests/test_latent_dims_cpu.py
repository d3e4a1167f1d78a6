"""Latent-size limits without a GPU: the entry points refuse shapes past their limits with RLCTR_EUNSUPPORTED and bad arguments
with RLCTR_EINVAL before any CUDA call, and the error raised for an unsupported shape states the limit."""
import ctypes as C

import pytest

from rl_ctr_prediction_b200 import _lib

EINVAL, EUNSUPPORTED = -1, -2
_FAKE = 1 << 20                     # 16-byte aligned stand-in address: every call below returns before reading through it


def _table(rs, lin, emb, dim, n_rows=1000):
    return _lib.Table(_FAKE, n_rows, rs, lin, emb, dim, 0)


def test_embed_rows_past_36_floats_are_refused():
    lib = _lib.load()
    for rs, lin, emb, dim in ((40, 0, 1, 33), (40, -1, 0, 40), (64, 0, 1, 60)):
        t = _table(rs, lin, emb, dim)
        assert lib.rlctr_embed_fwd(_FAKE, C.byref(t), None, _FAKE, None, 1, None, None, 0, 64, 15, 0, None) == EUNSUPPORTED
    t = _table(36, 0, 1, 40)                                                      # latent columns past the row
    assert lib.rlctr_embed_fwd(_FAKE, C.byref(t), None, _FAKE, None, 1, None, None, 0, 64, 15, 0, None) == EINVAL
    t = _table(36, 0, 1, 32)
    assert lib.rlctr_embed_fwd(_FAKE, C.byref(t), None, _FAKE, None, 1, None, None, 0, -1, 15, 0, None) == EINVAL
    assert lib.rlctr_embed_fwd(_FAKE, C.byref(t), None, _FAKE, None, 1, None, _FAKE, 100, 64, 15, 0, None) == EINVAL  # rows pitch


def test_afm_past_d32_is_refused():
    lib = _lib.load()
    for D in (33, 64):
        assert lib.rlctr_afm_fwd(_FAKE, 15 * D, _FAKE, _FAKE, 64, 15, D, 0.0, None, None, None) == EUNSUPPORTED
        assert lib.rlctr_afm_bwd(_FAKE, 15 * D, _FAKE, _FAKE, _FAKE, 15 * D, _FAKE, 64, 15, D, 0.0, None, None, _FAKE, 1 << 30,
                                 None) == EUNSUPPORTED
    assert lib.rlctr_afm_fwd(_FAKE, 24 * 8, _FAKE, _FAKE, 64, 24, 8, 0.0, None, None, None) == EUNSUPPORTED      # F > 23
    assert lib.rlctr_afm_fwd(_FAKE, 15 * 32, _FAKE, _FAKE, 64, 15, 0, 0.0, None, None, None) == EINVAL
    assert lib.rlctr_afm_fwd(_FAKE, 15 * 32 - 1, _FAKE, _FAKE, 64, 15, 32, 0.0, None, None, None) == EINVAL        # ld_rows < F*D
    assert lib.rlctr_afm_fwd(_FAKE, 15 * 32, _FAKE, _FAKE, 64, 15, 32, 0.2, None, None, None) == EINVAL           # p > 0, no rng
    assert lib.rlctr_afm_fwd(_FAKE, 15 * 32, _FAKE, _FAKE, 64, 15, 32, 1.0, _FAKE, None, None) == EINVAL
    assert lib.rlctr_afm_bwd(_FAKE, 15 * 32, _FAKE, _FAKE, _FAKE, 15 * 32, _FAKE, 64, 15, 32, 0.0, None, None, _FAKE, 16,
                             None) == -3                                                                        # workspace


def test_cross_past_512_columns_is_refused():
    lib = _lib.load()
    for fd in (513, 1024):
        assert lib.rlctr_cross_fwd(_FAKE, fd, _FAKE, _FAKE, 5, _FAKE, fd, _FAKE, 64, fd, None) == EUNSUPPORTED
        assert lib.rlctr_cross_bwd(_FAKE, fd, _FAKE, _FAKE, _FAKE, 5, _FAKE, fd, _FAKE, fd, _FAKE, _FAKE, 64, fd, _FAKE, 1 << 30,
                                   None) == EUNSUPPORTED
    assert lib.rlctr_cross_fwd(_FAKE, 480, _FAKE, _FAKE, 9, _FAKE, 480, _FAKE, 64, 480, None) == EUNSUPPORTED       # layers > 8
    assert lib.rlctr_cross_fwd(_FAKE, 479, _FAKE, _FAKE, 5, _FAKE, 480, _FAKE, 64, 480, None) == EINVAL            # ldx < dim
    assert lib.rlctr_cross_bwd(_FAKE, 480, _FAKE, _FAKE, _FAKE, 5, _FAKE, 480, _FAKE, 480, _FAKE, _FAKE, 64, 480, _FAKE, 16,
                               None) == -3


def test_row_update_past_512_floats_is_refused():
    lib = _lib.load()
    t = _lib.Table(_FAKE, 1000, 516, 15 * 34, 0, 15 * 34, 3 * 516)                 # FFM, F = 15, D = 34: 511 + 1 -> 516 floats
    a = _lib.Adam(_FAKE, _FAKE, _FAKE, _FAKE, _FAKE, 8192, -1, 0.9, 0.999, 1e-8, 1e-5)
    g = _lib.RowGrad(_FAKE, _FAKE, None, None, 15, _lib.RLCTR_STAGED_PARTNER)
    assert lib.rlctr_rows_adam(_FAKE, _FAKE, 64, C.byref(g), C.byref(t), C.byref(a), _FAKE, 1 << 20, None) == EUNSUPPORTED
    assert lib.rlctr_rows_adam(_FAKE, _FAKE, -1, C.byref(g), C.byref(t), C.byref(a), _FAKE, 1 << 20, None) == EINVAL


def test_unsupported_shape_error_states_the_limit():
    lib = _lib.load()
    with pytest.raises(_lib.RlctrError, match=r"D <= 32, F <= 23"):
        _lib.call("rlctr_afm_fwd", lib.rlctr_afm_fwd, _FAKE, 15 * 40, _FAKE, _FAKE, 64, 15, 40, 0.0, None, None, None)
    with pytest.raises(_lib.RlctrError, match=r"F\*D <= 512"):
        _lib.call("rlctr_cross_fwd", lib.rlctr_cross_fwd, _FAKE, 600, _FAKE, _FAKE, 5, _FAKE, 600, _FAKE, 64, 600, None)
    t = _table(40, 0, 1, 33)
    with pytest.raises(_lib.RlctrError, match=r"at most 36 floats"):
        _lib.call("rlctr_embed_fwd", lib.rlctr_embed_fwd, _FAKE, C.byref(t), None, _FAKE, None, 1, None, None, 0, 64, 15, 0, None,
                  key="rlctr_embed_fwd[FM]")
    with pytest.raises(_lib.RlctrError, match=r"invalid argument") as e:                  # other codes carry no limit
        _lib.call("rlctr_afm_fwd", lib.rlctr_afm_fwd, None, 15 * 40, _FAKE, _FAKE, 64, 15, 40, 0.0, None, None, None)
    assert "supported:" not in str(e.value)
