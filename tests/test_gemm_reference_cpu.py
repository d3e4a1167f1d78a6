"""The exact-operand oracle, the planner mirror and the dropout port of test_gpu_gemm_edges.py, checked without a GPU: the operand
generators of every case meet the exactness precondition; a numpy emulation of 3xTF32 (hi by truncation and by rounding to tf32,
random k-orders, random split-K partitions) reproduces the fp64 result bit for bit on both exact families, and a dropped or doubled
k-block, a lost lo term, a shifted bias column or two swapped output rows each change it (so the GPU comparisons can fail); the
cases reach every planner branch in REQUIRED and the docstring's table is current; the constants the mirror copies still appear in
the sources; the workspace mirror matches rlctr_mlp_ws_bytes; and the dropout port's one-key fast path equals its per-element
formula at every alignment and at the 2^32 pair crossing."""
import os
import re

import numpy as np
import pytest

import test_gpu_gemm_edges as G


# ---------------------------------------------------------------------------------------------------------------------------
# 3xTF32 in numpy
# ---------------------------------------------------------------------------------------------------------------------------
def tf32_trunc(x):
    return (np.asarray(x, np.float32).view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)


def tf32_rn(x):
    with np.errstate(over="ignore"):
        return ((np.asarray(x, np.float32).view(np.uint32) + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)


def emulate(A, Bm, bias, hi, rng, splits=1, drop_block=None, double_block=None, drop_lo=False):
    """C = A Bm^T + bias as the kernels compute it: (hi, lo) split of both operands, the tensor core reading each as tf32
    (truncation), three fp32 products per k accumulated in fp32 in a random k-order inside each split, the split partials added
    in order, then the bias."""
    A, Bm = np.asarray(A, np.float32), np.asarray(Bm, np.float32)
    Ah, Bh = hi(A), hi(Bm)
    Al, Bl = tf32_trunc(A - Ah), tf32_trunc(Bm - Bh)
    K = A.shape[1]
    kb = (K + G.BK - 1) // G.BK
    blocks = [list(range(b * G.BK, min(K, (b + 1) * G.BK))) for b in range(kb)]
    if drop_block is not None:
        blocks[drop_block] = []
    if double_block is not None:
        blocks.append(list(blocks[double_block]))
    cuts = np.sort(rng.choice(np.arange(1, len(blocks)), size=splits - 1, replace=False)) if splits > 1 else []
    parts = np.split(np.arange(len(blocks)), cuts)
    out = np.zeros((A.shape[0], Bm.shape[0]), np.float32)
    for part in parts:
        ks = [k for b in part for k in blocks[b]]
        ks = [ks[i] for i in rng.permutation(len(ks))]
        acc = np.zeros_like(out)
        for k in ks:
            terms = [np.outer(Ah[:, k], Bh[:, k])]
            if not (drop_lo and Al[:, k].any()):
                terms.append(np.outer(Al[:, k], Bh[:, k]))
            if not (drop_lo and Bl[:, k].any()):
                terms.append(np.outer(Ah[:, k], Bl[:, k]))
            for t in terms:
                acc = (acc + t.astype(np.float32)).astype(np.float32)
        out = (out + acc).astype(np.float32)
    return (out + np.asarray(bias, np.float32)).astype(np.float32)


def family(fam, M, K, N, seed, scale=1.0):
    """fwd-shaped operands of a family, the streamed one scaled by `scale` (1.25: the ReLU + dropout backward's gy_scale)"""
    A, Bm, b = G.fwd_operands(fam, M, K, N, seed)
    return (A * np.float32(scale)).astype(np.float32), Bm, b


@pytest.mark.parametrize("scale", [1.0, 1.25])
@pytest.mark.parametrize("fam", ["A", "B"])
@pytest.mark.parametrize("hi", [tf32_rn, tf32_trunc], ids=["hi_rn", "hi_trunc"])
@pytest.mark.parametrize("seed", range(3))
def test_3xtf32_emulation_is_exact_on_both_families(seed, hi, fam, scale):
    A, Bm, b = family(fam, 24, 100 + seed, 20, seed)
    s, lim = G.exact_window(A, Bm, b)
    assert s < lim
    ref = A.astype(np.float64) @ Bm.astype(np.float64).T + b
    assert np.array_equal(ref.astype(np.float32).astype(np.float64), ref)           # fp32 holds the exact result
    rng = np.random.default_rng(seed)
    for splits in (1, 2, 4):
        got = emulate(A, Bm, b, hi, rng, splits)
        assert np.array_equal(got, ref.astype(np.float32)), (splits, np.abs(got - ref).max())


@pytest.mark.parametrize("fam", ["A", "B"])
@pytest.mark.parametrize("mutation", ["drop_block", "double_block", "drop_lo", "shift_bias", "swap_rows"])
def test_oracle_rejects_a_wrong_gemm(fam, mutation):
    A, Bm, b = family(fam, 24, 100, 20, 7)
    ref = (A.astype(np.float64) @ Bm.astype(np.float64).T + b).astype(np.float32)
    rng = np.random.default_rng(1)
    if mutation == "drop_block":
        got = emulate(A, Bm, b, tf32_rn, rng, drop_block=1)
    elif mutation == "double_block":
        got = emulate(A, Bm, b, tf32_rn, rng, double_block=2)
    elif mutation == "drop_lo":
        got = emulate(A, Bm, b, tf32_rn, rng, drop_lo=True)
    elif mutation == "shift_bias":
        got = emulate(A, Bm, np.roll(b, 1), tf32_rn, rng)
    else:
        got = emulate(A, Bm, b, tf32_rn, rng)[[1, 0] + list(range(2, A.shape[0]))]
    assert not np.array_equal(got, ref)


def test_plain_tf32_is_not_exact():
    """the families do carry a lo part that a single tf32 product would lose"""
    for fam in ("A", "B"):
        A, Bm, b = family(fam, 24, 100, 20, 3)
        ref = (A.astype(np.float64) @ Bm.astype(np.float64).T + b).astype(np.float32)
        one = (tf32_trunc(A).astype(np.float64) @ tf32_trunc(Bm).astype(np.float64).T + b).astype(np.float32)
        assert not np.array_equal(one, ref)


# ---------------------------------------------------------------------------------------------------------------------------
# every case's operands meet the precondition
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fam", ["A", "B"])
@pytest.mark.parametrize("case", G.FWD_CASES + G.DROP_CASES, ids=lambda c: c.name)
def test_fwd_generators_meet_the_precondition(case, fam):
    x, w, b = G.fwd_inputs(case, fam)
    s, lim = G.exact_window(x, w, b)
    assert s < lim <= 2.0 ** 10, (s, lim)


@pytest.mark.parametrize("relu", [0, 1])
@pytest.mark.parametrize("fam", ["A", "B"])
@pytest.mark.parametrize("case", G.BWD_CASES, ids=lambda c: c.name)
def test_bwd_generators_meet_the_precondition(case, fam, relu):
    x, w, dy, y, dy_eff, _, _ = G.bwd_inputs(case, fam, relu)
    for s, lim in G.bwd_windows(x, w, dy_eff):
        assert s < lim, (s, lim)
    assert (dy_eff != 0).mean() > 0.5 * G.bwd_density(case.B, case.N) * (0.5 if relu else 1) * (2 / 3 if fam == "B" else 1)


# ---------------------------------------------------------------------------------------------------------------------------
# planner mirror: coverage, docstring table, source constants, workspace
# ---------------------------------------------------------------------------------------------------------------------------
def reached():
    labs = set()
    for c in G.FWD_CASES + G.BWD_CASES:
        labs |= G.branches(c)
    for c in G.DROP_CASES:
        for ctr in G.counters(c.N).values():
            labs |= G.drop_branches(c, ctr)
    return labs


def test_cases_reach_every_branch():
    missing = G.REQUIRED - reached()
    assert not missing, sorted(missing)


def test_docstring_table_is_current():
    assert G.table() in G.__doc__


def test_case_names_are_unique():
    names = [c.name for c in G.FWD_CASES + G.BWD_CASES + G.DROP_CASES]
    assert len(names) == len(set(names))


@pytest.mark.parametrize("fname,pattern,what", G.SOURCE_CONSTANTS, ids=[w for _, _, w in G.SOURCE_CONSTANTS])
def test_mirrored_constants_appear_in_the_sources(fname, pattern, what):
    with open(os.path.join(G.CSRC, fname)) as f:
        assert re.search(pattern, f.read()), (fname, what, pattern)


@pytest.fixture(scope="module")
def lib():
    from rl_ctr_prediction_b200 import _lib
    return _lib.load()


def test_workspace_mirror_matches_the_library(lib):
    """rlctr_mlp_ws_bytes sizes the dW partials from both planners' split counts: the mirror's splits must agree"""
    shapes = {(c.B, c.K, c.N) for c in G.FWD_CASES + G.BWD_CASES}
    shapes |= {(B, K, N) for B in (1, 31, 33, 4095, 4097, 65535) for K in (1, 31, 150, 600) for N in (1, 2, 75, 300)}
    for B, K, N in sorted(shapes):
        assert lib.rlctr_mlp_ws_bytes(B, K, N) == G.ws_layout(B, K, N)["total"], (B, K, N)


def test_mirror_matches_the_hand_computed_plans():
    """the plans the issue-level edges rely on, written out"""
    p = G.tma_plan(304, 36, 40001, True, True, True)
    last = p["kb"] - (p["splits"] - 1) * p["kps"]
    assert (p["splits"], p["kps"], last, 40001 % 32) == (49, 26, 3, 1)
    p = G.tma_plan(18945, 36, 300, True, False, True)
    assert p["n_tile"] == 64 and p["stages"] == 6 and not p["c_tma"] and p["tiles"] == 149
    p = G.tma_plan(129, 200, 8, False, False, True)
    assert p["n_tile"] == 112 and p["c_tma"] and p["n_tiles"] == 2
    p = G.tma_plan(18944, 300, 150, False, False, True)
    assert p["tiles"] == 2 * G.SMS
    p = G.tma_plan(200, 152, 300, True, True, True)
    assert p["splits"] == 1 and p["c_tma"]
    p = G.tma_plan(1024, 1024, 1100, True, True, False)
    assert (p["n_tiles"], p["splits"]) == (7, 2)


# ---------------------------------------------------------------------------------------------------------------------------
# dropout port
# ---------------------------------------------------------------------------------------------------------------------------
def test_dropout_fast_path_equals_per_element_formula():
    seed, thr = G.SEED, G.dropout_thresh(0.2)
    starts = [0, 2, 30, 62, 1 << 20, (1 << 32) - 64, (1 << 33) - 64, (1 << 33) + 2, (1 << 40) + 6]
    for w in (16, 32):
        for i0 in starts:
            for a in range(0, 64, 2):                      # every even alignment of the chunk start
                j = i0 + a
                if (j >> 33) != ((j + w - 1) >> 33):
                    continue
                want = G.keep(seed, np.arange(j, j + w, dtype=np.uint64), thr)
                assert np.array_equal(G.keep_chunk_fast(seed, j, w, thr), want), (w, j)


def test_dropout_pair_crossing_needs_the_per_element_formula():
    """a chunk whose pair index crosses 2^32 spans two keys: the one-key formula would be wrong there, which is why the epilogue
    takes the per-element path; and the per-element formula changes key exactly at element 2^33"""
    seed, thr = G.SEED, G.dropout_thresh(0.5)
    for w in (16, 32):
        j = (1 << 33) - 8
        idx = np.arange(j, j + w, dtype=np.uint64)
        want = G.keep(seed, idx, thr)
        p0 = j >> 1
        key = G.dropout_key(seed, np.uint32(p0 >> 32))
        h = G.dropout_bits(key, ((np.uint64(p0) + np.arange(w // 2, dtype=np.uint64)) & np.uint64(0xFFFFFFFF)).astype(np.uint32))
        one_key = np.empty(w, bool)
        one_key[0::2] = (h & np.uint32(0xFFFF)) >= thr
        one_key[1::2] = (h >> np.uint32(16)) >= thr
        assert np.array_equal(one_key[:8], want[:8]) and not np.array_equal(one_key, want)


def test_dropout_port_statistics_and_constants():
    seed = G.SEED
    idx = np.arange(1 << 18, dtype=np.uint64) + np.uint64(12345)
    for p in (0.2, 0.5):
        k = G.keep(seed, idx, G.dropout_thresh(p))
        assert abs(k.mean() - (1 - p)) < 0.005
    assert G.dropout_thresh(0.2) == 13107 and G.dropout_thresh(0.5) == 32768
    assert G.dropout_scale(0.5) == np.float32(2.0) and G.dropout_scale(0.2) == np.float32(1.25)
    # the odd counter puts every fused chunk of an even-N case on the per-element path, N = 75 every other row
    c = G.DROP_CASES[0]
    assert "drop:slow_every_row" in G.drop_branches(c, G.counters(c.N)["odd"])
    assert "drop:slow_odd_rows" in G.drop_branches(G.DROP_CASES[2], 0)
    for c in G.DROP_CASES[:3]:
        assert "drop:slow_pair_crossing" in G.drop_branches(c, G.counters(c.N)["cross2^33"])


def test_dropout_port_matches_the_cuda_source():
    """the hash constants of common.cuh are the port's"""
    with open(os.path.join(G.CSRC, "common.cuh")) as f:
        src = f.read()
    for const in ("0x7feb352dU", "0x846ca68bU", "0x9e3779b9U"):
        assert const in src
    assert "x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;" in src
    assert "return ((idx & 1) ? (h >> 16) : (h & 0xffffu)) >= thresh;" in src
