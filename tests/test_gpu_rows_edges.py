"""The sparse Adam row update (csrc/optim.cu) on every dispatch branch, at the run-length, tile and grid edges, against an fp64
reference with per-element error bounds.

Reference: the per-occurrence gradients of a step are built in float64 from the same fp32 inputs the kernel reads (FM rows:
dz * (S - v) with v the row the kernel gathered) and scattered with ``np.add.at``; Adam is ``np_oracle.adam_step(...,
dtype=np.float64)`` -- the reference's dense ``torch.optim.Adam`` with L2 folded into the gradient.  A row that missed steps is
first replayed in float64 through those steps with a zero data gradient.  Every row is checked against a bound carried through
the same step (``adam_bounded_step``): a row with L occurrences may carry an fp32 sum error of (L + 4) * 2^-24 * sum_i |g_i| (the
terms of every g_i counted by absolute value), which (1 - beta1) carries into exp_avg and (1 - beta2) * 2|g| into exp_avg_sq; a
few ulp of each new value cover the roundings of the step itself, and a parameter may move by a few ulp of itself, 16 ulp of its
update (the SFU square root and reciprocals, the fp32 schedule) and lr times the relative error of its moments.  Untouched rows,
padding columns, the gap between the p / exp_avg / exp_avg_sq blocks of a record and NaN-filled guard rows past n_rows are checked
bit for bit, and every case is run twice and must give the same bits.

Case -> kernel it reaches (launch_rows / rlctr_group_rows_adam in csrc/optim.cu; RLCTR_ROWS_R and RLCTR_ROWS_GRID are read once
per process, so their non-default values run in child processes, ``test_cached_switch``):

    case             geometry (row_stride, used, stamp)            entry            kernels
    scalar_lr        rs 1, no state in the record, stamp array     rows_adam        rows_scalar_kernel<0>
    scalar_lr_stage  rs 1, [w|m|v|stamp] records                   lookup+rows_adam rows_scalar_kernel<0> (from the stage)
    stage_rs4        rs 4, used 3, stamp in record                 lookup+rows_adam rows_staged_kernel<1,4> + rows_long<1,0>
    stage_rs8        rs 8, used 6                                  lookup+rows_adam rows_staged_kernel<2,4> + rows_long<2,0>
    tile_c1..c4      rs 16, used 3 / 6 / 11 / 15                   lookup+rows_adam rows_staged_tile_kernel<C> + rows_long<4,0>
    short_rs4        rs 4, used 4, stamp array                     rows_adam        rows_short<1,0> + rows_long<1,0>
    short_rs8        rs 8, used 8, stamp array                     rows_adam        rows_short<2,0> + rows_long<2,0>
    short_rs16       rs 16, used 16, stamp array                   rows_adam        rows_short<4,0> + rows_long<4,0>
    short_rs32       rs 32, used 31, stamp array                   rows_adam        rows_short<8,0> + rows_long<8,0>
    wide_fm36        rs 36 (FM D = 32), stamp array                rows_adam        rows_wide_kernel<0,2>
    wide_ffm272      rs 272 (FFM F = 15, D = 18), stamp array      rows_adam        rows_wide_kernel<0,4>
    group_rows2_3    rs 24, 6 chunks, one member per chunk         group_rows_adam  group_rows2_kernel<3> + rows_long<8,0,true,512>
    group_rows2_4    rs 28, 7 chunks                               group_rows_adam  group_rows2_kernel<4> + rows_long<8,0,true,512>
    group_eight_env  group_rows2_3's layout, RLCTR_GROUP_ROWS2=0   group_rows_adam  rows_short<8,0,true> + rows_long<8,0,true,512>
    group_eight_shr  rs 24, two members share a chunk              group_rows_adam  rows_short<8,0,true> + rows_long<8,0,true,512>
    group_four       rs 12 (lanes per row 4)                       group_rows_adam  rows_short<4,0,true> + rows_long<4,0,true>
    group_wide16_l1  rs 24, a member at lanes-per-row 8            group_rows_adam  rows_short<16,0,true> + group_long_wide
    group_wide16_l2  rs 44, two lines (max_lines 2)                group_rows_adam  rows_short<16,0,true> + group_long_wide
    group_wide32_l4  rs 92, three lines, members at lpr 16 / 8,   group_rows_adam  rows_short<32,0,true> + group_long_wide
                     a tail member's extra at extra_pitch > dim
    dense_*          the rows_adam geometries above                rows_grad_dense  rows_scalar<1> / rows_short<L,1> +
                                                                                    rows_long<L,1> / rows_wide<1,2|4>

Catch-up and flush (``test_replay_*``): rows_catchup_scalar_kernel / adam_flush_scalar_kernel (LR records), replay_kernel<true|false>
+ catchup_stamp_kernel / stamp_fill_kernel (separate stamps), replay_rows_kernel<CH, LPRR> at 1-, 2- and 4-line records, and
rlctr_rows_catchup_ids' claim-bit kernel over duplicate batch-order ids.
"""
import ctypes as C
import os
import subprocess
import sys
from dataclasses import dataclass, field

import numpy as np
import pytest
import torch

from oracle import np_oracle as O

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
U = 2.0 ** -24                          # unit roundoff of fp32
B1, B2, EPS, WD, LR = 0.9, 0.999, 1e-8, 1e-3, 1e-3
GUARD = 8                               # NaN-filled rows past n_rows in every table, moment and gradient array
STAMP_GUARD = -7
TILE, LONG_RUN = 128, 32                # csrc/optim.cu: tile::TT and LONG_RUN


# ---------------------------------------------------------------------------------------------------------------------------
# id streams: run lengths in sorted-id order (+ out-of-range ids, sorted last); every generator names the edge it places
# ---------------------------------------------------------------------------------------------------------------------------
@dataclass
class Stream:
    name: str
    lengths: np.ndarray                  # run lengths of the in-range ids, in sorted id order
    n_rows: int
    n_oob: int = 0                       # out-of-range ids (sorted last)
    last_row: bool = False               # the last in-range run is on row n_rows - 1
    heads: list = field(default_factory=list)       # sorted positions the generator claims are run heads
    runs: list = field(default_factory=list)        # run lengths the generator claims occur

    @property
    def n(self):
        return int(self.lengths.sum()) + self.n_oob


def _from_heads(heads, n):
    """Run lengths whose heads are exactly `heads` (0 included) in a sorted view of n in-range positions."""
    h = np.array(sorted(set([0] + list(heads))), np.int64)
    return np.diff(np.append(h, n))


def stream_runs():
    rng = np.random.default_rng(1)
    want = [1, 2, 31, 32, 33, 34, 64, 65, 128, 129]
    lengths = np.array(want * 3 + [1] * 7, np.int64)
    rng.shuffle(lengths)
    return Stream("runs_1_to_129", lengths, 2000, runs=want)


def stream_tile_heads():
    heads = []
    for j in range(1, 9):
        heads += [TILE * j - 1, TILE * j, TILE * j + 1]
    heads += [TILE * 9 - 16, TILE * 9 + 17]                    # a run of 33 straddling a tile boundary
    heads += [TILE * 10 + 95, TILE * 10 + 128]                 # a run of 33 whose 32-id look-ahead ends on the tile's last slot
    heads += [TILE * 11 + 96, TILE * 11 + 128]                 # a run of 32 whose look-ahead is the next tile's first id
    heads += [TILE * 12 - 1, TILE * 12 + 32]                   # a run of 33 from the last slot of a tile
    n = TILE * 13 + 5
    return Stream("tile_heads", _from_heads(heads, n), 3000, heads=sorted(heads), runs=[33, 32])


def stream_one_id(n):
    return Stream(f"one_id_n{n}", np.array([n], np.int64), 700, heads=[0], runs=[n])


def stream_many_long():
    return Stream("400_runs_of_40", np.full(400, 40, np.int64), 5000, runs=[40])


def stream_zipf(n=200_003, n_rows=50_000):
    rng = np.random.default_rng(7)
    ids = np.minimum(rng.zipf(1.2, size=n) - 1, n_rows - 1)
    lengths = np.bincount(ids, minlength=n_rows)
    lengths = lengths[lengths > 0]
    rng.shuffle(lengths)
    return Stream(f"zipf_{n}", lengths, n_rows)


def stream_oob_tail():
    lengths = np.array([3, 1, 40, 2, 33, 1, 50], np.int64)
    return Stream("oob_after_last_row", lengths, 900, n_oob=40, last_row=True, runs=[50])


def stream_ragged():
    rng = np.random.default_rng(3)
    lengths = rng.integers(1, 6, size=600)
    lengths[-1] += 1 + (-int(lengths.sum())) % 8                 # n = 1 (mod 8): not a multiple of 8 or of 128
    return Stream("ragged_n_odd", lengths, 4000)


def all_streams(zipf=True):
    s = [stream_runs(), stream_tile_heads()] + [stream_one_id(n) for n in (1, 32, 33, 4096)]
    s += [stream_many_long(), stream_oob_tail(), stream_ragged()]
    if zipf:
        s.append(stream_zipf())
    return s


STREAMS = {s.name: s for s in all_streams()}


def draw(stream, rng):
    """A batch of ids (batch order) whose sorted view has the stream's runs: distinct random rows, shuffled positions."""
    N, k = stream.n_rows, len(stream.lengths)
    pool = N - 1 if stream.last_row else N
    rows = np.sort(rng.choice(pool, size=k - stream.last_row, replace=False))
    if stream.last_row:
        rows = np.append(rows, N - 1)
    view = np.repeat(rows.astype(np.int64), stream.lengths)
    oob = np.array([N, N + 1, N + 77, -1, 1 << 40], np.int64)[np.arange(stream.n_oob) % 5]
    view = np.concatenate([view, oob])
    return view[rng.permutation(view.size)]


def sorted_view(ids, n_rows):
    """What rlctr_sort_ids produces: ids (out-of-range -> n_rows) stably sorted, and their batch positions."""
    key = np.where((ids >= 0) & (ids < n_rows), ids, n_rows)
    order = np.argsort(key, kind="stable")
    return key[order], order


# ---------------------------------------------------------------------------------------------------------------------------
# fp64 reference with per-element bounds
# ---------------------------------------------------------------------------------------------------------------------------
def sched_row(t, lr=LR):
    return O.adam_schedule(t, lr, B1, B2)


def adam_bounded_step(P, M, V, Bp, Bm, Bv, G, Bg, t, lr=LR, wd=WD):
    """One fp64 Adam step (np_oracle.adam_step) of state (P, M, V) with gradient G, and the bounds (Bp, Bm, Bv) an fp32 kernel
    that started within (Bp, Bm, Bv) of the state and summed G within Bg stays within after it."""
    P1, M1, V1 = O.adam_step(P, G, M, V, t, lr, wd, B1, B2, EPS, dtype=np.float64)
    g = G + wd * P
    bg = Bg + wd * Bp + 2 * U * np.abs(g)
    bm = Bm + (1 - B1) * bg + 4 * U * ((1 - B1) * np.abs(g - M) + np.abs(M1))
    bv = B2 * Bv + (1 - B2) * (2 * np.abs(g) * bg + bg * bg) + 4 * U * ((1 - B2) * g * g + B2 * np.abs(V) + np.abs(V1))
    ss, bc2 = sched_row(t, lr)
    denom = np.sqrt(V1) / bc2 + EPS
    upd = ss * M1 / denom
    with np.errstate(divide="ignore", invalid="ignore"):             # |sqrt(a) - sqrt(b)| = |a - b| / (sqrt(a) + sqrt(b))
        dden = np.where(V1 > 0, bv / (np.sqrt(V1) + np.sqrt(np.maximum(V1 - bv, 0))), np.sqrt(bv)) / bc2
        rel = np.where(dden < denom, dden / (denom - dden), np.inf)
    bp = Bp + 4 * U * np.abs(P1) + 16 * U * np.abs(upd) + ss * bm / denom + np.abs(upd) * rel + ss * bm * rel / denom
    return P1, M1, V1, bp, bm, bv


def replay(P, M, V, stamps, upto, lr=LR, wd=WD):
    """fp64 dense Adam with a zero data gradient from each row's stamp to `upto`, with the bounds an fp32 replay stays within."""
    P, M, V = (np.asarray(a, np.float64).copy() for a in (P, M, V))
    Bp, Bm, Bv = np.zeros_like(P), np.zeros_like(P), np.zeros_like(P)
    stamps = np.asarray(stamps)
    if stamps.size == 0:
        return P, M, V, Bp, Bm, Bv
    state = (P, M, V, Bp, Bm, Bv)
    for t in range(int(stamps.min()) + 1, upto + 1):
        live = np.nonzero(stamps < t)[0]
        zero = np.zeros((live.size, P.shape[1]))
        out = adam_bounded_step(*(x[live] for x in state[:3]), *(x[live] for x in state[3:]), zero, zero, t, lr, wd)
        for x, y in zip(state, out):
            x[live] = y
    return state


def within(got, want, bound):
    """Per-element |got - want| <= bound (an element with bound 0 must be exact)."""
    got = np.asarray(got, np.float64)
    return np.isfinite(got) & (np.abs(got - want) <= bound)


def assert_within(got, want, bound, what):
    ok = within(got, want, bound)
    if not ok.all():
        i = np.argwhere(~ok)[:4]
        raise AssertionError(f"{what}: {int((~ok).sum())} of {ok.size} elements out of bound; first at {i.tolist()}: "
                             f"got {[float(np.asarray(got)[tuple(j)]) for j in i]}, want {[float(want[tuple(j)]) for j in i]}, "
                             f"bound {[float(bound[tuple(j)]) for j in i]}")


def occurrence_grads(view_ids, view_slots, uniq, p_rows, comp):
    """Dense per-row gradient (fp64) and sum_i |terms of g_i| over the occurrences, by np.add.at.  comp(slot, p) -> list of
    [n_occ, rs] float64 terms of each occurrence's gradient; p: the gathered row of the occurrence's id."""
    pos = np.searchsorted(uniq, view_ids)
    terms = comp(view_slots, p_rows[pos])
    G = np.zeros((uniq.size, p_rows.shape[1]))
    A = np.zeros_like(G)
    gsum = terms[0].copy()
    for x in terms[1:]:
        gsum += x
    np.add.at(G, pos, gsum)
    np.add.at(A, pos, sum(np.abs(x) for x in terms))
    return G, A


# ---------------------------------------------------------------------------------------------------------------------------
# cases
# ---------------------------------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Case:
    name: str
    rs: int
    lin: int
    emb: int
    dim: int
    entry: str = "rows"                 # rows | staged | group | dense
    stamp: str = "array"                # array | record
    record: bool = True                 # [p | exp_avg | exp_avg_sq] records (pitch 3 * block)
    block: int = 0                      # floats per block of a record (0: rs)
    stamp_at: int = -1
    members: tuple = ()                 # group: (lin, emb, dim, fm_term, extra_pitch or 0 = no extra)
    env: tuple = ()                     # per-call switches: (name, value)

    @property
    def used(self):
        if self.members:
            return self.stamp_at
        return max(self.lin + 1, self.emb + self.dim, 1)


def _group(name, rs, members, stamp_at, env=()):
    blk = 32 if rs <= 32 else rs
    return Case(name, rs, -1, 0, stamp_at, "group", "record", True, blk, stamp_at, tuple(members), env)


FM, TAIL = True, False
CASES = [
    Case("scalar_lr", 1, 0, 0, 0, record=False),
    Case("scalar_lr_stage", 1, 0, 0, 0, "staged", "record"),
    Case("stage_rs4", 4, 0, 1, 2, "staged", "record"),
    Case("stage_rs8", 8, 0, 1, 5, "staged", "record"),
    Case("tile_c1", 16, 0, 1, 2, "staged", "record"),
    Case("tile_c2", 16, 0, 1, 5, "staged", "record"),
    Case("tile_c3", 16, 0, 1, 10, "staged", "record"),
    Case("tile_c4", 16, 0, 1, 14, "staged", "record"),
    Case("short_rs4", 4, 0, 1, 3),
    Case("short_rs8", 8, 0, 1, 7),
    Case("short_rs16", 16, 0, 1, 15),
    Case("short_rs32", 32, 0, 1, 30),
    Case("wide_fm36", 36, 0, 1, 32),
    Case("wide_ffm272", 272, 270, 0, 270),
    # joint records: members (lin, emb, dim, FM term, extra pitch); LR members are (col, 0, 0, False, 0)
    _group("group_rows2_3", 24, [(0, 1, 10, FM, 0), (12, 13, 10, FM, 10), (11, 0, 0, FM, 0)], 23),
    _group("group_rows2_4", 28, [(0, 1, 10, FM, 0), (12, 13, 14, FM, 14), (11, 0, 0, FM, 0)], 27),
    _group("group_eight_env", 24, [(0, 1, 10, FM, 0), (12, 13, 10, FM, 10), (11, 0, 0, FM, 0)], 23, (("RLCTR_GROUP_ROWS2", "0"),)),
    _group("group_eight_shr", 24, [(0, 1, 5, FM, 0), (-1, 6, 6, TAIL, 6), (12, 13, 7, FM, 7), (20, 0, 0, FM, 0)], 21),
    _group("group_four", 12, [(0, 1, 6, FM, 0), (7, 0, 0, FM, 0)], 9),
    _group("group_wide16_l1", 24, [(0, 1, 20, FM, 20), (21, 0, 0, FM, 0)], 22),
    _group("group_wide16_l2", 44, [(0, 1, 10, FM, 0), (12, 13, 10, FM, 10), (-1, 24, 16, TAIL, 16), (11, 0, 0, FM, 0)], 41),
    _group("group_wide32_l4", 92, [(0, 1, 32, FM, 0), (36, 37, 30, FM, 30), (-1, 68, 20, TAIL, 25), (33, 0, 0, FM, 0)], 89),
    Case("dense_scalar", 1, 0, 0, 0, "dense", record=False),
    Case("dense_rs4", 4, 0, 1, 3, "dense"),
    Case("dense_rs8", 8, 0, 1, 7, "dense"),
    Case("dense_rs16", 16, 0, 1, 15, "dense"),
    Case("dense_rs32", 32, 0, 1, 30, "dense"),
    Case("dense_fm36", 36, 0, 1, 32, "dense"),
    Case("dense_ffm272", 272, 270, 0, 270, "dense"),
]
CASE = {c.name: c for c in CASES}


def lib():
    from rl_ctr_prediction_b200 import _lib
    return _lib.load()


def L():
    from rl_ctr_prediction_b200 import _lib
    return _lib


def ptr(t):
    return None if t is None else t.data_ptr()


def stream_handle():
    return torch.cuda.current_stream().cuda_stream


def gpu_sort(ids_d, n_rows):
    n = ids_d.numel()
    sid = torch.empty(n, dtype=torch.int32, device=DEV)
    ss = torch.empty(n, dtype=torch.int32, device=DEV)
    wsb = lib().rlctr_sort_ws_bytes(n, n_rows)
    ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
    assert lib().rlctr_sort_ids(ptr(ids_d), n, n_rows, ptr(sid), ptr(ss), ptr(ws), wsb, stream_handle()) == 0
    return sid, ss


class Harness:
    """A table with guard rows, its Adam state and the checks around one call of the update."""

    def __init__(self, case, n_rows, seed, sched_len=1024, check=True):
        from rl_ctr_prediction_b200.tables import AdamSchedule, Geometry
        c = self.case = case
        self.check = check                               # False: run the calls only (the determinism rerun)
        self.N = N = n_rows
        rng = self.rng = np.random.default_rng(seed)
        rs, used = c.rs, c.used
        blk = c.block or rs
        self.blk = blk
        if c.record:
            pitch = 4 if rs == 1 else 3 * blk
            if c.members and rs > 32:
                pitch = (3 * rs + 31) // 32 * 32
            self.geom = Geometry(N, rs, c.lin, c.emb, c.dim, pitch, c.block, c.stamp_at)
        else:
            pitch = rs
            self.geom = Geometry(N, rs, c.lin, c.emb, c.dim)
        self.stamp_col = self.geom.stamp_col if c.stamp == "record" else -1
        assert (self.stamp_col >= 0) == (c.stamp == "record"), (c.name, self.stamp_col)
        self.pitch = pitch
        tab = np.full((N + GUARD, pitch), np.nan, np.float32)
        state = np.zeros((N, rs), np.float32)
        state[:, :used] = rng.standard_normal((N, used)) * 0.3
        if c.members:                                    # a stamp column or padding inside `used` carries no parameter
            state[:, self.owned_mask() == 0] = 0
        mom = np.zeros((N, rs), np.float32)
        vel = np.zeros((N, rs), np.float32)
        mom[:, :used] = rng.standard_normal((N, used)) * 1e-3     # nonzero moments: the parameter check then sees g itself
        vel[:, :used] = rng.uniform(1e-7, 1e-6, (N, used))
        if c.members:
            mom[:, self.owned_mask() == 0] = 0
            vel[:, self.owned_mask() == 0] = 0
        if 0 <= self.stamp_col < rs:                    # (LR records keep it past the row: [w | m | v | stamp])
            state[:, self.stamp_col] = 0; mom[:, self.stamp_col] = 0; vel[:, self.stamp_col] = 0
        if c.record:
            mb, vb = (1, 2) if rs == 1 else (blk, 2 * blk)
            tab[:N, :rs] = state
            tab[:N, mb:mb + rs] = mom
            tab[:N, vb:vb + rs] = vel
            self.tab = torch.as_tensor(tab).to(DEV)
            self.m_off, self.v_off = mb, vb
            self.m = self.v = None
        else:
            self.tab = torch.as_tensor(tab).to(DEV)
            self.tab[:N] = torch.as_tensor(state).to(DEV)
            mm = np.full((N + GUARD, rs), np.nan, np.float32); mm[:N] = mom
            vv = np.full((N + GUARD, rs), np.nan, np.float32); vv[:N] = vel
            self.m, self.v = torch.as_tensor(mm).to(DEV), torch.as_tensor(vv).to(DEV)
        if self.stamp_col >= 0:
            self.tab[:N, self.stamp_col] = 0.0
            self.stamp = None
        else:
            st = np.full(N + GUARD, STAMP_GUARD, np.int32); st[:N] = 0
            self.stamp = torch.as_tensor(st).to(DEV)
        self.step = torch.zeros(1, dtype=torch.int32, device=DEV)
        self.sched = AdamSchedule(LR, (B1, B2), torch.device(DEV), sched_len).tensor
        self.keep = []

    # -- layout --------------------------------------------------------------------------------------------------------
    def owned_mask(self):
        """Per column of the row: 0 no parameter, 1 first-order weight, 2 latent with the FM term, 3 latent without."""
        c = self.case
        role = np.zeros(c.rs, np.int8)
        if c.members:
            for lin, emb, dim, fm, _ in c.members:
                if lin >= 0:
                    role[lin] = 1
                role[emb:emb + dim] = 2 if fm else 3
        else:
            if c.lin >= 0:
                role[c.lin] = 1
            role[c.emb:c.emb + c.dim] = np.where(np.arange(c.emb, c.emb + c.dim) == c.lin, 1, 2)
            if c.rs == 1:
                role[0] = 1
        return role

    def struct(self, stage=None):
        t = L().Table(self.tab.data_ptr(), self.N, self.case.rs, self.case.lin, self.case.emb, self.case.dim, self.pitch)
        if self.case.record:
            m, v = self.tab.data_ptr() + 4 * self.m_off, self.tab.data_ptr() + 4 * self.v_off
        else:
            m, v = self.m.data_ptr(), self.v.data_ptr()
        a = L().Adam(m, v, ptr(self.stamp), ptr(self.sched), ptr(self.step), self.sched.shape[0], self.stamp_col, B1, B2, EPS, WD,
                     ptr(stage))
        return t, a

    def snapshot(self):
        """(p, m, v) [N + GUARD, rs] fp32 and stamps [N + GUARD] as numpy, and the raw record bits."""
        tab = self.tab.cpu().numpy()
        rs = self.case.rs
        if self.case.record:
            p, m, v = tab[:, :rs], tab[:, self.m_off:self.m_off + rs], tab[:, self.v_off:self.v_off + rs]
        else:
            p, m, v = tab, self.m.cpu().numpy(), self.v.cpu().numpy()
        if self.stamp_col >= 0:
            stamps = tab[:, self.stamp_col].view(np.int32)
        else:
            stamps = self.stamp.cpu().numpy()
        bits = [tab.view(np.int32).copy()] + ([] if self.case.record else [self.m.cpu().numpy().view(np.int32),
                                                                           self.v.cpu().numpy().view(np.int32)])
        return p.copy(), m.copy(), v.copy(), stamps.copy(), bits

    # -- gradient inputs -----------------------------------------------------------------------------------------------
    def grad_inputs(self, n, F):
        """dL/dlogit per sample, column sums S per sample (NaN where no FM term reads them), per-occurrence staged rows and
        dense-tail rows."""
        c, rng = self.case, self.rng
        B = n // F
        role = self.owned_mask()
        inp = {"F": F, "dz": (rng.standard_normal(B) * 0.05).astype(np.float32)}
        S = np.full((B, c.rs), np.nan, np.float32)
        S[:, role == 2] = rng.standard_normal((B, int((role == 2).sum()))) * 0.3
        inp["S"] = S if (role == 2).any() else None
        if c.members:
            inp["dzm"] = [(rng.standard_normal(B) * 0.05).astype(np.float32) for _ in c.members]
            ex = []
            for lin, emb, dim, fm, xp in c.members:
                if xp:
                    e = np.full((n, xp), np.nan, np.float32)
                    e[:, :dim] = rng.standard_normal((n, dim)) * 0.01
                    ex.append(e)
                else:
                    ex.append(None)
            inp["extra"] = ex
        else:
            stg = np.zeros((n, c.rs), np.float32)
            stg[:, role > 0] = rng.standard_normal((n, int((role > 0).sum()))) * 0.01
            inp["staged"] = stg
            if c.dim and c.rs > 1 and c.rs <= 32:
                inp["ex"] = (rng.standard_normal((n, c.dim)) * 0.01).astype(np.float32)
        return inp

    def comp_fn(self, inp):
        """terms of each occurrence's gradient, [n_occ, rs] float64 each (the same fp32 inputs as the kernel)."""
        c, F = self.case, inp["F"]
        role = self.owned_mask()

        def comp(slots, p):
            b = slots // F
            f = slots - b * F
            p = p.astype(np.float64)
            terms = []
            if c.members:
                for (lin, emb, dim, fm, xp), dzm, ex in zip(c.members, inp["dzm"], inp["extra"]):
                    t = np.zeros_like(p)
                    dz = dzm[b].astype(np.float64)
                    if lin >= 0:
                        t[:, lin] = dz
                    cols = np.arange(emb, emb + dim)
                    if fm and dim:
                        t[:, cols] = dz[:, None] * (inp["S"][b][:, cols].astype(np.float64) - p[:, cols])
                    terms.append(t)
                    if ex is not None:
                        e = np.zeros_like(p)
                        e[:, cols] = ex[slots, :dim]
                        terms.append(e)
                return terms
            terms.append(inp["staged"][slots].astype(np.float64))
            dz = np.zeros_like(p)
            dz[:, role == 1] = inp["dz"][b].astype(np.float64)[:, None]
            terms.append(dz)
            if inp["S"] is not None:
                t = np.zeros_like(p)
                cols = np.nonzero(role == 2)[0]
                t[:, cols] = inp["dz"][b].astype(np.float64)[:, None] * (inp["S"][b][:, cols].astype(np.float64) - p[:, cols])
                terms.append(t)
            if inp.get("ex") is not None:
                t = np.zeros_like(p)
                t[:, c.emb:c.emb + c.dim] = inp["ex"].reshape(-1, F, c.dim)[b, f]
                terms.append(t)
            return terms
        return comp

    def rowgrad(self, inp):
        d = lambda x: None if x is None else self._dev(x)
        if self.case.rs == 1:
            return L().RowGrad(ptr(d(inp["staged"])), ptr(d(inp["dz"])), None, None, inp["F"], 0)
        return L().RowGrad(ptr(d(inp["staged"])), ptr(d(inp["dz"])), ptr(d(inp["S"])), ptr(d(inp.get("ex"))), inp["F"], 0)

    def _dev(self, x):
        t = torch.as_tensor(np.ascontiguousarray(x)).to(DEV)
        self.keep.append(t)
        return t

    # -- one step ------------------------------------------------------------------------------------------------------
    def step_once(self, ids, F, s, where):
        """Step s (the device step counter is s - 1) on a batch of ids: the case's entry point, then every check."""
        c, N, rs = self.case, self.N, self.case.rs
        n = ids.size
        ids_d = self._dev(ids)
        sid, ss = gpu_sort(ids_d, N)
        view_ids, view_slots = sorted_view(ids, N)
        assert np.array_equal(sid.cpu().numpy().astype(np.int64), view_ids), f"{where}: sorted view"
        inr = view_ids < N
        vid, vslot = view_ids[inr], view_slots[inr]
        uniq, heads = np.unique(vid, return_index=True)
        counts = np.diff(np.append(heads, vid.size))
        inp = self.grad_inputs(n, F)
        p0, m0, v0, st0, bits0 = self.snapshot()
        role = self.owned_mask()
        act = role > 0
        lazy = self.stamp_col >= 0 or self.stamp is not None
        wsb = lib().rlctr_rows_ws_bytes(n)
        ws = self._dev(np.zeros(wsb, np.uint8))
        if c.entry == "dense":
            dense = self._dev(np.full((N + GUARD, rs), np.nan, np.float32))
            t, _ = self.struct()
            g = self.rowgrad(inp)
            assert lib().rlctr_rows_grad_dense(ptr(sid), ptr(ss), n, C.byref(g), C.byref(t), ptr(dense), ptr(ws), wsb,
                                               stream_handle()) == 0
            if not self.check:
                return
            G, A = occurrence_grads(vid, vslot, uniq, p0[uniq], self.comp_fn(inp))
            got = dense.cpu().numpy()
            Bg = (counts[:, None] + 4) * U * A
            assert_within(got[uniq], G, Bg, f"{where}: dense gradient")
            rest = np.ones(N + GUARD, bool); rest[uniq] = False
            assert np.isnan(got[rest]).all(), f"{where}: dense gradient written outside the batch's rows"
            assert np.array_equal(self.snapshot()[4][0], bits0[0]), f"{where}: the table changed"
            return
        # pre-step state of the touched rows: the stored record replayed to s - 1 (lazy) in fp64
        if self.check:
            P, M, V, Bp, Bm, Bv = replay(p0[uniq], m0[uniq], v0[uniq], st0[uniq] if lazy else np.full(uniq.size, s - 1), s - 1)
        pg = p0[uniq]                                    # the row the kernel's gradient sees
        if c.entry == "staged":
            t, a = self.struct()
            sf = lib().rlctr_lookup_stage_floats(C.byref(t))
            stage = self._dev(np.full(n * sf, np.nan, np.float32))
            gathered = self._dev(np.zeros((n, rs), np.float32))
            lk = L().Lookup(ptr(stage), 0, 0)
            lk.gathered[0] = ptr(gathered)
            rc = lib().rlctr_rows_lookup(ptr(sid), ptr(ss), n, C.byref(t), C.byref(a), C.byref(lk), ptr(ws), wsb, stream_handle())
            assert rc == 0, lib().rlctr_strerror(rc)
            sg = stage.cpu().numpy().reshape(n, sf)[heads] if self.check else np.zeros((uniq.size, sf), np.float32)
            if rs == 1:
                sp, sm, sv = sg[:, 0:1], sg[:, 1:2], sg[:, 2:3]
            else:
                bs = sf // 3
                pad = lambda x: np.concatenate([x, np.zeros((x.shape[0], rs - bs), np.float32)], axis=1) if rs > bs else x
                sp, sm, sv = pad(sg[:, :bs]), pad(sg[:, bs:2 * bs]), pad(sg[:, 2 * bs:])
            for got, want, bnd, nm in ((sp, P, Bp, "p"), (sm, M, Bm, "exp_avg"), (sv, V, Bv, "exp_avg_sq")) if self.check else ():
                assert_within(got[:, act], want[:, act], bnd[:, act], f"{where}: staged {nm} (lookup replay)")
            P, M, V = sp.astype(np.float64), sm.astype(np.float64), sv.astype(np.float64)
            Bp, Bm, Bv = np.zeros_like(P), np.zeros_like(P), np.zeros_like(P)
            pg = sp
            t, a = self.struct(stage)
            g = self.rowgrad(inp)
            rc = lib().rlctr_rows_adam(ptr(sid), ptr(ss), n, C.byref(g), C.byref(t), C.byref(a), ptr(ws), wsb, stream_handle())
        elif c.entry == "rows":
            t, a = self.struct()
            g = self.rowgrad(inp)
            rc = lib().rlctr_rows_adam(ptr(sid), ptr(ss), n, C.byref(g), C.byref(t), C.byref(a), ptr(ws), wsb, stream_handle())
        else:
            t, a = self.struct()
            arr = (L().Member * len(c.members))()
            for i, (lin, emb, dim, fm, xp) in enumerate(c.members):
                arr[i].lin_col, arr[i].emb_col, arr[i].dim = lin, emb, dim
                arr[i].flags = L().RLCTR_FM_TERM if fm else 0
                arr[i].dlogit = ptr(self._dev(inp["dzm"][i]))
                arr[i].extra = ptr(self._dev(inp["extra"][i])) if xp else None
                arr[i].extra_pitch = xp if (xp and xp != dim) else 0
            sums = self._dev(inp["S"])
            rc = lib().rlctr_group_rows_adam(ptr(sid), ptr(ss), n, C.byref(t), C.byref(a), arr, len(c.members), ptr(sums), 0,
                                             F, 1, None, ptr(ws), wsb, stream_handle())
        assert rc == 0, lib().rlctr_strerror(rc)
        assert lib().rlctr_step_advance(ptr(self.step), 1, stream_handle()) == 0
        torch.cuda.synchronize()
        if not self.check:
            return
        G, A = occurrence_grads(vid, vslot, uniq, pg, self.comp_fn(inp))
        Bg = (counts[:, None] + 4) * U * A
        P1, M1, V1, Bp1, Bm1, Bv1 = adam_bounded_step(P, M, V, Bp, Bm, Bv, G, Bg, s)
        p1, m1, v1, st1, bits1 = self.snapshot()
        assert_within(m1[uniq][:, act], M1[:, act], Bm1[:, act], f"{where}: exp_avg")
        assert_within(v1[uniq][:, act], V1[:, act], Bv1[:, act], f"{where}: exp_avg_sq")
        assert_within(p1[uniq][:, act], P1[:, act], Bp1[:, act], f"{where}: parameters")
        pad = ~act
        if 0 <= self.stamp_col < rs:                    # LR records keep the stamp past the row: [w | m | v | stamp]
            pad[self.stamp_col] = False
        for x, nm in ((p1, "p"), (m1, "exp_avg"), (v1, "exp_avg_sq")):
            assert not x[uniq][:, pad].view(np.int32).any(), f"{where}: padding columns of {nm} not zero"
        if lazy:
            assert (st1[uniq] == s).all(), f"{where}: stamps of the touched rows"
        # untouched rows and guard rows, bit for bit (whole records: stamps, padding and block gaps included)
        rest = np.ones(N + GUARD, bool); rest[uniq] = False
        for b0, b1 in zip(bits0, bits1):
            assert np.array_equal(b0[rest], b1[rest]), f"{where}: rows outside the batch changed"
            ext = np.ones(b0.shape[1], bool); ext[:rs] = False
            if self.stamp_col >= 0:
                ext[self.stamp_col] = False
            if self.case.record:
                ext[self.m_off:self.m_off + rs] = False; ext[self.v_off:self.v_off + rs] = False
                assert np.array_equal(b0[uniq][:, ext], b1[uniq][:, ext]), f"{where}: record columns outside the blocks changed"
        if self.stamp is not None:
            assert (st1[N:] == STAMP_GUARD).all(), f"{where}: guard stamps"

    def state(self):
        p, m, v, st, bits = self.snapshot()
        return bits + [st.view(np.int32)]


def fields_for(n):
    for F in (15, 7, 5, 3):
        if n % F == 0:
            return F
    return 1


def run_case(case_name, stream_name, steps=3, seed=0, check=True):
    """All steps of one case on one stream, checked after every step (`check`); returns the final state bits."""
    c, s = CASE[case_name], STREAMS[stream_name]
    for k, v in c.env:
        os.environ[k] = v
    try:
        h = Harness(c, s.n_rows, seed, check=check)
        rng = np.random.default_rng(seed + 1)
        for step in range(1, steps + 1):
            ids = draw(s, rng)
            h.step_once(ids, fields_for(ids.size), step, f"{case_name} / {stream_name} / step {step}")
        torch.cuda.synchronize()
        return h.state()
    finally:
        for k, _ in c.env:
            os.environ.pop(k, None)


# Each case runs on every edge stream; the Zipf stream (several grid passes) on the cases with a persistent or tiled grid.
ZIPF_CASES = {"scalar_lr", "scalar_lr_stage", "stage_rs4", "tile_c3", "short_rs16", "short_rs32", "group_rows2_3",
              "group_eight_env", "group_four", "group_wide16_l1", "group_wide32_l4", "dense_rs16", "wide_fm36"}
EDGE_STREAMS = [s.name for s in all_streams(zipf=False)]
ZIPF = stream_zipf().name
PAIRS = [(c.name, s) for c in CASES for s in EDGE_STREAMS] + [(c, ZIPF) for c in sorted(ZIPF_CASES)]


@pytest.fixture(scope="module", autouse=True)
def _built():
    lib()


@pytest.mark.parametrize("case,stream", PAIRS)
def test_rows_edges(case, stream):
    steps = 2 if stream == ZIPF else 3
    a = run_case(case, stream, steps)
    b = run_case(case, stream, steps, check=False)
    for x, y in zip(a, b):
        assert np.array_equal(x, y), f"{case} / {stream}: not bit-identical from run to run"


# ---------------------------------------------------------------------------------------------------------------------------
# switches read once per process: one child process per value
# ---------------------------------------------------------------------------------------------------------------------------
SWITCH_RUNS = {
    # RLCTR_ROWS_R != 0: the phased kernel at lanes per row 4 as well; 2: two rows per lane group
    ("RLCTR_ROWS_R", "1"): ["stage_rs4", "stage_rs8", "tile_c2", "tile_c4"],
    ("RLCTR_ROWS_R", "2"): ["stage_rs4", "stage_rs8", "tile_c2", "tile_c4"],
    # RLCTR_ROWS_GRID 0: one block per group of positions; 2: twice the persistent grid
    ("RLCTR_ROWS_GRID", "0"): ["short_rs16", "short_rs32", "group_rows2_3", "group_eight_env", "group_wide16_l2", "dense_rs8"],
    ("RLCTR_ROWS_GRID", "2"): ["short_rs16", "short_rs32", "group_rows2_3", "group_eight_env", "group_wide16_l2", "dense_rs8"],
}


def child_main(cases, streams):
    for c in cases:
        for s in streams:
            a = run_case(c, s, 2)
            b = run_case(c, s, 2, check=False)
            assert all(np.array_equal(x, y) for x, y in zip(a, b)), f"{c} / {s}: not bit-identical from run to run"
    print("child ok")


@pytest.mark.parametrize("var,value", list(SWITCH_RUNS))
def test_cached_switch(var, value):
    here = os.path.dirname(os.path.abspath(__file__))
    root = os.path.dirname(here)
    cases = SWITCH_RUNS[(var, value)]
    streams = ["tile_heads", "400_runs_of_40", "oob_after_last_row", ZIPF]
    code = (f"import sys; sys.path[:0] = [{here!r}, {root!r}]; import test_gpu_rows_edges as t; "
            f"t.child_main({cases!r}, {streams!r})")
    env = dict(os.environ)
    env[var] = value
    args = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", code]
    r = subprocess.run(args, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "child ok" in r.stdout, f"{var}={value}:\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}"


# ---------------------------------------------------------------------------------------------------------------------------
# catch-up and flush: fp64 dense Adam with zero gradient and weight decay over the rows each call covers
# ---------------------------------------------------------------------------------------------------------------------------
REPLAY_CASES = {
    "lr_record": Case("lr_record", 1, 0, 0, 0, "rows", "record"),
    "fm16_record": Case("fm16_record", 16, 0, 1, 10, "rows", "record"),
    "fm16_array": Case("fm16_array", 16, 0, 1, 15),
    "group_1line": _group("group_1line", 24, [(0, 1, 10, FM, 0), (12, 13, 10, FM, 0), (11, 0, 0, FM, 0)], 23),
    "group_2line": _group("group_2line", 52, [(0, 1, 20, FM, 0), (24, 25, 24, FM, 0), (21, 0, 0, FM, 0)], 49),
    "group_4line": _group("group_4line", 112, [(0, 1, 32, FM, 0), (36, 37, 30, FM, 0), (-1, 68, 40, TAIL, 0)], 109),
}
STALENESS = (0, 1, 2, 300)


@pytest.mark.parametrize("entry", ["catchup", "catchup_ids", "flush"])
@pytest.mark.parametrize("geom", list(REPLAY_CASES))
def test_replay(geom, entry):
    if entry == "catchup_ids" and geom != "group_1line":
        pytest.skip("rlctr_rows_catchup_ids serves joint records of 5..8 chunks")
    c = REPLAY_CASES[geom]
    N, now = 3001, 310
    results = []
    for rep in range(2):
        h = Harness(c, N, seed=5, sched_len=1024)
        rng = np.random.default_rng(9)
        stamps = now - np.array(STALENESS)[rng.integers(0, len(STALENESS), N)]
        if h.stamp_col >= 0:
            h.tab[:N, h.stamp_col] = torch.as_tensor(stamps.astype(np.int32).view(np.float32)).to(DEV)
        else:
            h.stamp[:N] = torch.as_tensor(stamps.astype(np.int32)).to(DEV)
        h.step.fill_(now)
        p0, m0, v0, st0, bits0 = h.snapshot()
        t, a = h.struct()
        if entry == "flush":
            r0, r1 = 37, N - 91                           # ends off every block and tile boundary
            rows = np.arange(r0, r1)
            assert lib().rlctr_adam_flush(C.byref(t), C.byref(a), r0, r1, stream_handle()) == 0
        else:
            ids = np.concatenate([rng.integers(0, N, 5000), np.full(40, 17), [N, N + 3, -1]]).astype(np.int64)
            rng.shuffle(ids)
            ids_d = h._dev(ids)
            rows = np.unique(ids[(ids >= 0) & (ids < N)])
            if entry == "catchup":
                sid, _ = gpu_sort(ids_d, N)
                assert lib().rlctr_rows_catchup(ptr(sid), ids.size, C.byref(t), C.byref(a), stream_handle()) == 0
            else:
                cb = lib().rlctr_rows_claim_bytes(N)
                claim = h._dev(np.zeros(cb, np.uint8))
                rc = lib().rlctr_rows_catchup_ids(ptr(ids_d), ids.size, C.byref(t), C.byref(a), ptr(claim), cb, stream_handle())
                assert rc == 0, lib().rlctr_strerror(rc)
        torch.cuda.synchronize()
        p1, m1, v1, st1, bits1 = h.snapshot()
        act = h.owned_mask() > 0
        P, M, V, Bp, Bm, Bv = replay(p0[rows], m0[rows], v0[rows], st0[rows], now)
        where = f"{geom} / {entry}"
        assert_within(m1[rows][:, act], M[:, act], Bm[:, act], f"{where}: exp_avg")
        assert_within(v1[rows][:, act], V[:, act], Bv[:, act], f"{where}: exp_avg_sq")
        assert_within(p1[rows][:, act], P[:, act], Bp[:, act], f"{where}: parameters")
        assert (st1[rows] == now).all(), f"{where}: stamps"
        pad = ~act
        if 0 <= h.stamp_col < c.rs:
            pad[h.stamp_col] = False
        assert not p1[rows][:, pad].view(np.int32).any(), f"{where}: padding columns"
        rest = np.ones(N + GUARD, bool); rest[rows] = False
        for b0, b1 in zip(bits0, bits1):
            assert np.array_equal(b0[rest], b1[rest]), f"{where}: rows outside the call changed"
        if h.stamp is not None:
            assert (st1[N:] == STAMP_GUARD).all(), f"{where}: guard stamps"
        results.append(h.state())
    for x, y in zip(*results):
        assert np.array_equal(x, y), f"{geom} / {entry}: not bit-identical from run to run"
