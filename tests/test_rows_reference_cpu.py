"""The fp64 row-update reference of test_gpu_rows_edges.py, checked without a GPU: it agrees with np_oracle's fp32 Adam within
fp32 rounding, its per-element bound rejects an update that dropped or doubled one occurrence of a run of 33 or used the wrong
step index (so the GPU checks can fail), and every id-stream generator places the runs and heads it claims."""
import numpy as np
import pytest

from oracle import np_oracle as O
from test_gpu_rows_edges import (LR, U, WD, adam_bounded_step, all_streams, draw, replay, sorted_view, within)

B1, B2, EPS = 0.9, 0.999, 1e-8


def _run(seed, L=33, rs=12, step=3):
    """A row with L occurrences of random gradients, fp32 state; returns inputs and the fp64 reference with its bounds."""
    rng = np.random.default_rng(seed)
    p = (rng.standard_normal((1, rs)) * 0.3).astype(np.float32)
    m = (rng.standard_normal((1, rs)) * 1e-3).astype(np.float32)
    v = rng.uniform(1e-7, 1e-6, (1, rs)).astype(np.float32)
    g = (rng.standard_normal((L, rs)) * 0.01).astype(np.float32)
    G = g.astype(np.float64).sum(axis=0, keepdims=True)
    Bg = (L + 4) * U * np.abs(g.astype(np.float64)).sum(axis=0, keepdims=True)
    z = np.zeros_like(G)
    ref = adam_bounded_step(p, m, v, z, z, z, G, Bg, step)
    return p, m, v, g, ref


def _fp32_update(p, m, v, g_rows, step):
    """An fp32 update as a kernel does it: the occurrences summed in fp32 in order, then fp32 Adam."""
    acc = np.zeros_like(p)
    for r in g_rows:
        acc = (acc + r).astype(np.float32)
    return O.adam_step(p, acc, m, v, step, LR, WD, B1, B2, EPS, dtype=np.float32)


@pytest.mark.parametrize("seed", range(6))
def test_reference_is_oracle_adam_in_fp64_and_fp32_adam_is_within_bound(seed):
    p, m, v, g, (P1, M1, V1, Bp, Bm, Bv) = _run(seed, L=1 + 7 * seed)
    G = g.astype(np.float64).sum(axis=0, keepdims=True)
    want = O.adam_step(p, G, m, v, 3, LR, WD, B1, B2, EPS, dtype=np.float64)
    for a, b in zip((P1, M1, V1), want):
        assert np.array_equal(a, b)
    p32, m32, v32 = _fp32_update(p, m, v, g, 3)
    assert within(m32, M1, Bm).all() and within(v32, V1, Bv).all() and within(p32, P1, Bp).all()


def test_replay_reference_is_oracle_adam_and_fp32_replay_is_within_bound():
    rng = np.random.default_rng(4)
    p = (rng.standard_normal((5, 8)) * 0.3).astype(np.float32)
    m = (rng.standard_normal((5, 8)) * 1e-3).astype(np.float32)
    v = rng.uniform(1e-7, 1e-6, (5, 8)).astype(np.float32)
    stamps = np.array([0, 1, 2, 40, 42])
    P, M, V, Bp, Bm, Bv = replay(p, m, v, stamps, 42)
    for i, st in enumerate(stamps):
        a, b, c = p[i:i + 1].astype(np.float64), m[i:i + 1].astype(np.float64), v[i:i + 1].astype(np.float64)
        x, y, z = p[i:i + 1], m[i:i + 1], v[i:i + 1]
        for t in range(st + 1, 43):
            a, b, c = O.adam_step(a, None, b, c, t, LR, WD, B1, B2, EPS, dtype=np.float64)
            x, y, z = O.adam_step(x, None, y, z, t, LR, WD, B1, B2, EPS, dtype=np.float32)
        assert np.array_equal(P[i:i + 1], a) and np.array_equal(M[i:i + 1], b) and np.array_equal(V[i:i + 1], c)
        assert within(x, a, Bp[i:i + 1]).all() and within(y, b, Bm[i:i + 1]).all() and within(z, c, Bv[i:i + 1]).all()


@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("mutation", ["dropped", "doubled", "step_off_by_one"])
def test_bound_rejects_a_miscounted_occurrence_or_step(seed, mutation):
    p, m, v, g, (P1, M1, V1, Bp, Bm, Bv) = _run(100 + seed)
    step = 3
    if mutation == "dropped":
        g = np.delete(g, 17, axis=0)
    elif mutation == "doubled":
        g = np.insert(g, 17, g[17], axis=0)
    else:
        step = 4
    p32, m32, v32 = _fp32_update(p, m, v, g, step)
    if mutation == "step_off_by_one":                    # the moments do not depend on the step index; the parameter does
        assert not within(p32, P1, Bp).all()
    else:
        assert not within(m32, M1, Bm).all() and not within(v32, V1, Bv).all()


@pytest.mark.parametrize("stream", all_streams(), ids=lambda s: s.name)
def test_stream_generators_place_their_runs(stream):
    ids = draw(stream, np.random.default_rng(0))
    assert ids.size == stream.n
    key, _ = sorted_view(ids, stream.n_rows)
    inr = key < stream.n_rows
    assert (~inr).sum() == stream.n_oob and not inr[int(inr.sum()):].any()
    rows, heads, counts = np.unique(key[inr], return_index=True, return_counts=True)
    assert np.array_equal(counts, stream.lengths)
    for h in stream.heads:
        assert h in set(heads.tolist()), (stream.name, h)
    for r in stream.runs:
        assert r in set(counts.tolist()), (stream.name, r)
    if stream.last_row:
        assert rows[-1] == stream.n_rows - 1 and counts[-1] == stream.lengths[-1]
    if stream.name == "tile_heads":                      # a run of 33 straddling a tile boundary
        assert any(h % 128 > 128 - 33 and c == 33 for h, c in zip(heads, counts))
    if stream.name.startswith("zipf"):
        assert stream.n > 3 * 148 * 128 and stream.n > 740 * 64         # several passes of the tile grid and the block grid
    if stream.name == "400_runs_of_40":
        assert (counts > 32).sum() > 148                                # more long runs than rows_long_kernel has blocks
    if stream.name == "ragged_n_odd":
        assert stream.n % 8 and stream.n % 128
