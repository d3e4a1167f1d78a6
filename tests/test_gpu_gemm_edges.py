"""The tower GEMMs (rlctr_linear_fwd / rlctr_linear_bwd: csrc/mlp_tma.cu, csrc/mlp.cu) on every planner and dispatch branch, at the
tile, split-K, pitch and dropout-counter edges, against exact fp64 results.

Exact-operand oracle.  One operand carries a low part, the other is a small integer: family "A" gives the streamed operand (x for
the forward call, dy for dgrad and wgrad) the values a + b * 2^-13 (a in {-1, 0, 1}, b in {-3 .. 3}) and the other operand
integers in {-1, 0, 1}; family "B" swaps the roles.  Bias is a multiple of 2^-13.  The (hi, lo) split of a + b * 2^-13 is exact
whether hi is rounded or truncated to tf32 (lo is a multiple of 2^-13 below 2^-10: at most 3 significant bits), and only one side
has a lo part, so the lo * lo product that 3xTF32 leaves out is zero and hi*hi + hi*lo + lo*hi is the exact product.  Every test
asserts the precondition sum_k |a_ik b_jk| + |bias_j| < 2^(23 - e) in fp64, with 2^-e the grid of the products (2^-13; 2^-15 once
the ReLU backward has scaled dy by 1.25).  Then every partial sum, in any order and any split-K partition, is a multiple of 2^-e that
fp32 holds exactly, and every path -- TMA, staged, simt, gemv, fused or elementwise epilogue -- must equal the fp64 result:
``torch.equal``, no tolerance.  A dropped, doubled or misplaced k-block, a tile at the wrong offset, a lost lo correction, a wrong
bias column or a wrong split partial shows up as a nonzero multiple of the grid step.  Dropout and mask scales multiply an exact
value once in fp32, which the reference repeats (``np.float32(v) * np.float32(1 / (1 - p))``).  On a B200 (sm_100a) the tcgen05
kind::tf32 MMAs held this as designed: every exact case passed at the full 2^10 window, no smaller window was needed.

Family "R" (random normal operands) checks precision instead: within 1e-5 of the output scale (plus 1e-5 of the element) of fp64,
and, except for dW, within 16x of fp32 SGEMM's own error (``check_precision`` says why dW is exempt).

Every case also checks, bit for bit: NaN sentinels in the 256 bytes before and after every output (y, dx, dW, db), which are views
into larger buffers, some of them 4 or 8 bytes off a 16-byte boundary; NaN in the rows past B of x and dy and in the pad columns
of a padded x; a NaN-filled workspace before every call (with RLCTR_MLP_W_PRESPLIT, all of it but the forward call's weight images);
x, w, bias and y unchanged, dy unchanged or, with RLCTR_MLP_RELU, equal to dy * (y > 0 ? gy_scale : 0); and the same bits on a second
run.  Dropout is checked against a numpy port of the counter hash of common.cuh (``keep``), bit for bit.

Case -> branches, from the mirror of make_plan (mlp_tma.cu), plan_gemm (mlp.cu) and the dispatch of rlctr_linear_fwd/bwd
(``python tests/test_gpu_gemm_edges.py`` prints it; tests/test_gemm_reference_cpu.py checks that this table is current and that the
cases reach every branch in REQUIRED):

    f_b1_k4               B 1 in 4 out 300                fwd:bias_smem fwd:c_tma fwd:k<32 fwd:n_tiles>1 fwd:tma
    f_b129_k8             B 129 in 8 out 200              fwd:bias_smem fwd:c_tma fwd:c_tma+tail16 fwd:k<32 fwd:n_tiles>1 fwd:tma
    f_two_tiles           B 18944 in 150 out 300 ldx 152  fwd:bias_smem fwd:c_tma fwd:cta_second_tile fwd:n_tiles>1 fwd:tma
    f_149_tiles           B 18945 in 1 out 16 ldx 4       fwd:bias_smem fwd:c_tma fwd:c_tma+tail16 fwd:cta_second_tile fwd:k<32 fwd:tma
    f_k33_n1100           B 300 in 33 out 1100 ldx 36     fwd:bias_global fwd:c_tma fwd:k%32==1 fwd:n_tiles>1 fwd:tma
    f_e32                 B 513 in 64 out 1030            fwd:bias_global fwd:cvec2 fwd:e32 fwd:n_tiles>1 fwd:tma
    f_e16                 B 999 in 100 out 75             fwd:bias_smem fwd:cvec1 fwd:e16 fwd:tma
    f_padded_y4           B 777 in 100 out 300 ldx 108    fwd:bias_smem fwd:cvec1 fwd:e32 fwd:n_tiles>1 fwd:tma
    f_y8                  B 300 in 64 out 200             fwd:bias_smem fwd:cvec2 fwd:e16 fwd:n_tiles>1 fwd:tma
    f_bench_150           B 65536 in 150 out 300 ldx 152  fwd:bias_smem fwd:c_tma fwd:cta_second_tile fwd:n_tiles>1 fwd:tma
    f_bench_300           B 65536 in 300 out 200          fwd:bias_smem fwd:c_tma fwd:c_tma+tail16 fwd:cta_second_tile fwd:n_tiles>1 fwd:tma
    f_x_misaligned        B 777 in 100 out 300            fwd:staged fwd:staged_n_tiles>1
    f_staged_env          B 300 in 33 out 1100            fwd:staged fwd:staged_n_tiles>1
    f_staged_e16          B 999 in 100 out 75             fwd:staged
    f_fp32_32             B 1000 in 150 out 300           fwd:simt32
    f_fp32_64             B 1024 in 64 out 1200           fwd:simt64
    f_gemv4               B 1000 in 152 out 1             fwd:gemv_rows4
    f_gemv_350            B 1000 in 350 out 1             fwd:gemv_rows
    f_gemv_680            B 1000 in 680 out 1             fwd:gemv_rows
    f_gemv_odd_ldx        B 1000 in 150 out 1 ldx 151     fwd:gemv_rows
    g_777_600_300         B 777 in 600 out 300            db:converter+reduce2 dgrad:c_tma dgrad:mask_tma dgrad:n_tiles>1 dgrad:tma wgrad:n_tiles>1_x_splits wgrad:splitk wgrad:tma
    g_777_600_300_nomask  B 777 in 600 out 300            dgrad:c_tma dgrad:n_tiles>1 dgrad:tma
    g_777_presplit        B 777 in 600 out 300            dgrad:c_tma dgrad:mask_tma dgrad:n_tiles>1 dgrad:presplit dgrad:tma
    g_1000_1100_64        B 1000 in 1100 out 64           db:colsum_kernel dgrad:c_tma dgrad:mask_tma dgrad:n_tiles>1 dgrad:tma
    g_18945_36_300        B 18945 in 36 out 300           dgrad:c_thread_smem dgrad:cta_second_tile dgrad:cvec4 dgrad:e32 dgrad:mask_thread dgrad:presplit dgrad:tma
    g_mask_pitch          B 777 in 600 out 300 ldx 601    db:colsum_kernel dgrad:c_tma dgrad:mask_thread dgrad:n_tiles>1 dgrad:tma wgrad:staged wgrad:staged_splitk
    g_dx_off4             B 777 in 600 out 300            dgrad:cvec1 dgrad:e32 dgrad:mask_thread dgrad:n_tiles>1 dgrad:tma
    g_out75               B 999 in 100 out 75             db:colsum_kernel dgrad:mask_rows_kernel dgrad:staged wgrad:staged wgrad:staged_splitk
    g_staged_env          B 777 in 600 out 300            db:colsum_kernel dgrad:mask_rows_kernel dgrad:staged wgrad:staged wgrad:staged_splitk
    g_fp32                B 1000 in 150 out 300           db:colsum_kernel dgrad:mask_rows_kernel dgrad:simt wgrad:simt
    w_300_152_200         B 300 in 152 out 200            db:converter+reduce dgrad:c_tma dgrad:tma wgrad:splits1_c_tma wgrad:tma
    w_dw_off8             B 300 in 152 out 200            db:converter+reduce wgrad:splits1_c_thread wgrad:tma
    w_2047_300_200        B 2047 in 300 out 200           db:converter+reduce2 wgrad:k%32==31 wgrad:n_tiles>1_x_splits wgrad:splitk wgrad:tma
    w_40001_36_304        B 40001 in 36 out 304           db:converter+reduce2 wgrad:short_last_split_one_row wgrad:splitk wgrad:tma
    w_1100_1024_1024      B 1100 in 1024 out 1024         db:converter+reduce2 wgrad:n_tiles>1_x_splits wgrad:splitk wgrad:tma
    w_ldx_odd             B 2047 in 300 out 200 ldx 301   db:colsum_kernel wgrad:staged wgrad:staged_splitk
    b_bench_150           B 65536 in 150 out 300 ldx 152  db:converter+reduce2 dgrad:cta_second_tile dgrad:cvec2 dgrad:e32 dgrad:presplit dgrad:tma wgrad:splitk wgrad:tma
    b_bench_300           B 65536 in 300 out 200          db:converter+reduce2 dgrad:c_tma dgrad:cta_second_tile dgrad:mask_tma dgrad:n_tiles>1 dgrad:presplit dgrad:tma wgrad:n_tiles>1_x_splits wgrad:splitk wgrad:tma
    o_150_all             B 1000 in 150 out 1 ldx 152     bwd1:colsum_parts bwd1:gemv_bwd8
    o_150_all_mask        B 1000 in 150 out 1             bwd1:colsum_parts bwd1:gemv_bwd8 bwd1:gemv_bwd_mask
    o_150_dx              B 1000 in 150 out 1             bwd1:gemv_bwd8
    o_150_dx_mask         B 1000 in 150 out 1             bwd1:gemv_bwd8 bwd1:gemv_bwd_mask
    o_150_dw              B 1000 in 150 out 1             bwd1:colsum_parts bwd1:gemv_bwd8
    o_150_db              B 1000 in 150 out 1             bwd1:colsum_parts bwd1:gemv_bwd8
    o_350_all             B 1000 in 350 out 1             bwd1:colsum_parts bwd1:gemv_bwd16
    o_350_all_mask        B 1000 in 350 out 1             bwd1:colsum_parts bwd1:gemv_bwd16 bwd1:gemv_bwd_mask
    o_350_dx              B 1000 in 350 out 1             bwd1:gemv_bwd16
    o_350_dx_mask         B 1000 in 350 out 1             bwd1:gemv_bwd16 bwd1:gemv_bwd_mask
    o_350_dw              B 1000 in 350 out 1             bwd1:colsum_parts bwd1:gemv_bwd16
    o_350_db              B 1000 in 350 out 1             bwd1:colsum_parts bwd1:gemv_bwd16
    o_680_all             B 1000 in 680 out 1             bwd1:colsum_db bwd1:colsum_dw bwd1:outer_rows
    o_680_all_mask        B 1000 in 680 out 1             bwd1:colsum_db bwd1:colsum_dw bwd1:outer_rows_mask
    o_680_dx              B 1000 in 680 out 1             bwd1:outer_rows
    o_680_dx_mask         B 1000 in 680 out 1             bwd1:outer_rows_mask
    o_680_dw              B 1000 in 680 out 1             bwd1:colsum_dw
    o_680_db              B 1000 in 680 out 1             bwd1:colsum_db
    d_c_tma               B 300 in 64 out 300             drop:fast drop:fused drop:pair_hi>0 drop:slow_every_row drop:slow_pair_crossing
    d_e32                 B 513 in 64 out 1030            drop:fast drop:fused drop:pair_hi>0 drop:slow_every_row drop:slow_pair_crossing
    d_e16                 B 999 in 100 out 75             drop:fast drop:fused drop:pair_hi>0 drop:slow_odd_rows drop:slow_pair_crossing
    d_kernel              B 300 in 64 out 300             drop:kernel drop:pair_hi>0
    d_kernel_75           B 999 in 100 out 75             drop:kernel drop:pair_hi>0
"""
import os
import sys
from dataclasses import dataclass

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "rl_ctr_prediction_b200", "csrc")

# ---------------------------------------------------------------------------------------------------------------------------
# mirror of the planners and the dispatch (every constant is checked against the sources by test_gemm_reference_cpu.py)
# ---------------------------------------------------------------------------------------------------------------------------
SMS = 148                 # common.cuh RLCTR_SMS
BM, BK = 128, 32          # mlp_tma.cu BM / BK; mlp.cu GEMM_BM / GEMM_BK
NT_MAX = 160              # mlp_tma.cu: widest TMA tile
TMEM_COLS = 512
MAX_STAGES = 8
SMEM_BUDGET = 220 * 1024  # pipeline + C staging (both planners)
MASK_BUDGET = 221 * 1024  # pipeline + C staging + dgrad mask blocks
BIAS_SMEM = 1024
C_STAGE_BYTES = 4 * 2 * 4096
M_STAGE_BYTES = 4 * 4096
STAGED_NT_MAX = 256       # mlp.cu plan_gemm: (N + 255) / 256
GEMV4_MAX = 256           # gemv_rows4_kernel and gemv_bwd_kernel<8>
GEMV_BWD_MAX = 512        # gemv_bwd_kernel<16>
COLSUM_ROWS = 128         # COLSUM_ROWS_PER_BLOCK

SOURCE_CONSTANTS = [      # (file, pattern that must appear, what it pins)
    ("common.cuh", rf"#define RLCTR_SMS {SMS}\b", "SMS"),
    ("mlp_tma.cu", rf"constexpr int BM = {BM};", "BM"),
    ("mlp_tma.cu", rf"constexpr int BK = {BK};", "BK"),
    ("mlp.cu", rf"constexpr int GEMM_BM = {BM};", "GEMM_BM"),
    ("mlp.cu", rf"constexpr int GEMM_BK = {BK};", "GEMM_BK"),
    ("mlp_tma.cu", rf"constexpr int NT_MAX = {NT_MAX};", "NT_MAX"),
    ("mlp_tma.cu", rf"constexpr int TMEM_COLS = {TMEM_COLS};", "TMEM_COLS"),
    ("mlp_tma.cu", rf"constexpr int MAX_STAGES = {MAX_STAGES};", "MAX_STAGES"),
    ("mlp.cu", rf"constexpr int GEMM_MAX_STAGES = {MAX_STAGES};", "GEMM_MAX_STAGES"),
    ("mlp_tma.cu", rf"constexpr int BIAS_SMEM = {BIAS_SMEM};", "BIAS_SMEM"),
    ("mlp_tma.cu", rf"\(size_t\)\({SMEM_BUDGET // 1024} \* 1024\) / stage_bytes", "TMA stage budget"),
    ("mlp_tma.cu", rf"C_STAGE_BYTES <= \(size_t\)\({SMEM_BUDGET // 1024} \* 1024\)", "C staging budget"),
    ("mlp_tma.cu", rf"M_STAGE_BYTES <= \(size_t\)\({MASK_BUDGET // 1024} \* 1024\)", "mask budget"),
    ("mlp_tma.cu", r"C_STAGE_BYTES = \(size_t\)EPI_WARPS \* 2 \* 4096", "C staging bytes"),
    ("mlp_tma.cu", r"M_STAGE_BYTES = \(size_t\)EPI_WARPS \* 4096", "mask staging bytes"),
    ("mlp_tma.cu", r"const int q = b_mn \? 32 : 16;", "tile quantum"),
    ("mlp_tma.cu", r"int max_s = kb_total / 8;", "k-blocks per split"),
    ("mlp.cu", rf"\(size_t\)\({SMEM_BUDGET // 1024} \* 1024\) / stage_bytes", "staged stage budget"),
    ("mlp.cu", rf"p.n_tiles = \(N \+ {STAGED_NT_MAX - 1}\) / {STAGED_NT_MAX};", "staged tile cap"),
    ("mlp.cu", r"int max_s = kb_total / 8;", "staged k-blocks per split"),
    ("mlp.cu", rf"in_dim % 4 == 0 && in_dim <= {GEMV4_MAX} && ldx % 4 == 0", "gemv_rows4 limit"),
    ("mlp.cu", rf"out_dim == 1 && in_dim <= {GEMV_BWD_MAX}\)", "gemv_bwd limit"),
    ("mlp.cu", rf"if \(in_dim <= {GEMV4_MAX}\)\n\s+gemv_bwd_kernel<8>", "gemv_bwd<8> limit"),
    ("mlp.cu", r"if \(big >= 2 \* RLCTR_SMS\)", "simt tile choice"),
    ("mlp.cu", rf"constexpr int COLSUM_ROWS_PER_BLOCK = {COLSUM_ROWS};", "colsum rows"),
]


def cdiv(a, b):
    return (a + b - 1) // b


def rup(n, q):
    return cdiv(n, q) * q


def tma_plan(M, N, K, b_mn, allow_split, c_ok):
    """make_plan of mlp_tma.cu"""
    q = 32 if b_mn else 16
    nts = cdiv(N, NT_MAX)
    nt = rup(cdiv(N, nts), q)
    mt = cdiv(M, BM)
    kb = cdiv(K, BK)
    s = 1
    if allow_split:
        s = min(max(SMS // max(mt * nts, 1), 1), max(kb // 8, 1))
    kps = max(cdiv(kb, s), 1)
    s = max(cdiv(kb, kps), 1)
    acc = rup(nt, 32)
    stage_bytes = BM * 128 + 2 * nt * 128
    st = min(SMEM_BUDGET // stage_bytes, MAX_STAGES, (TMEM_COLS - 2 * acc) // (2 * BK))
    c_tma = c_ok and s == 1 and stage_bytes * st + C_STAGE_BYTES <= SMEM_BUDGET
    smem = stage_bytes * st + (C_STAGE_BYTES if c_tma else 0) + 1024
    return dict(n_tile=nt, n_tiles=nts, m_tiles=mt, kb=kb, splits=s, kps=kps, stages=st, c_tma=c_tma, smem=smem,
                tiles=mt * nts * s)


def staged_plan(M, N, K, allow_split):
    """plan_gemm of mlp.cu"""
    nts = cdiv(N, STAGED_NT_MAX)
    nt = max(rup(cdiv(N, nts), 16), 16)
    mt = cdiv(M, BM)
    kb = cdiv(K, BK)
    s = 1
    if allow_split:
        s = min(max(SMS // max(mt * nts, 1), 1), max(kb // 8, 1))
    kps = max(cdiv(kb, s), 1)
    s = max(cdiv(kb, kps), 1)
    return dict(n_tile=nt, n_tiles=nts, m_tiles=mt, splits=s, kps=kps, tiles=mt * nts * s)


def align256(b):
    return (b + 255) & ~255


def ws_layout(B, K, N):
    """mlp_ws of mlp.cu: [split-K partials of dW | column-sum partials | W_hi | W_lo], bytes"""
    splits = max(staged_plan(N, K, B, True)["splits"], tma_plan(N, K, B, True, True, False)["splits"])
    wgrad = align256(splits * N * K * 4)
    colsum = align256(cdiv(B, COLSUM_ROWS) * (N + (K if N == 1 else 0)) * 4)
    wsplit = align256(N * rup(K, 4) * 4)
    return dict(wgrad=wgrad, colsum=colsum, wsplit=wsplit, images=wgrad + colsum, total=wgrad + colsum + 2 * wsplit + 256)


def vec_of(off, pitch):
    """widest aligned vector store of an output `off` floats past a 16-byte boundary"""
    if pitch % 4 == 0 and off % 4 == 0:
        return 4
    if pitch % 2 == 0 and off % 2 == 0:
        return 2
    return 1


def tma_ok(off, pitch):
    return off % 4 == 0 and pitch % 4 == 0


@dataclass
class Case:
    name: str
    op: str                   # "fwd" | "bwd"
    B: int
    K: int                    # in_dim
    N: int                    # out_dim
    ldx: int = 0              # 0: K
    x_off: int = 0            # x starts this many floats past a 16-byte boundary
    out_off: int = 0          # every output starts this many floats past a 16-byte boundary
    tma: bool = True          # RLCTR_GEMM_TMA
    fp32: bool = False        # RLCTR_MLP_FP32
    dx_mask: bool = False     # RLCTR_MLP_DX_MASK
    presplit: bool = False    # RLCTR_MLP_W_PRESPLIT (the forward call leaves the weight images in the workspace)
    want: str = "dx,dw,db"
    note: str = ""

    def __post_init__(self):
        self.ldx = self.ldx or self.K

    def wants(self, what):
        return what in self.want.split(",")


def _tma_labels(pre, p, M, N, K, bias, out_off, ldc):
    s = {f"{pre}:tma"}
    if p["tiles"] > SMS:
        s.add(f"{pre}:cta_second_tile")
    if p["n_tiles"] > 1:
        s.add(f"{pre}:n_tiles>1")
    if K < BK:
        s.add(f"{pre}:k<32")
    elif K % BK == 1:
        s.add(f"{pre}:k%32==1")
    elif K % BK == BK - 1:
        s.add(f"{pre}:k%32==31")
    if p["c_tma"]:
        s.add(f"{pre}:c_tma")
        if p["n_tile"] % 32:
            s.add(f"{pre}:c_tma+tail16")
    else:
        s.add(f"{pre}:e32" if p["n_tile"] % 32 == 0 else f"{pre}:e16")
        if p["splits"] == 1:
            s.add(f"{pre}:cvec{vec_of(out_off, ldc)}")
            if tma_ok(out_off, ldc):
                s.add(f"{pre}:c_thread_smem")
    if bias:
        s.add(f"{pre}:bias_smem" if p["n_tiles"] * p["n_tile"] <= BIAS_SMEM else f"{pre}:bias_global")
    return s


def fwd_plan(c):
    """(path, plan) of rlctr_linear_fwd"""
    if c.N == 1:
        ok4 = c.K % 4 == 0 and c.K <= GEMV4_MAX and c.ldx % 4 == 0 and c.x_off % 4 == 0
        return ("gemv_rows4" if ok4 else "gemv_rows"), None
    if c.fp32:
        return ("simt64" if cdiv(c.N, 64) * cdiv(c.B, 64) >= 2 * SMS else "simt32"), None
    if c.tma and tma_ok(c.x_off, c.ldx):
        return "tma", tma_plan(c.B, c.N, c.K, False, False, tma_ok(c.out_off, c.N))
    return "staged", staged_plan(c.B, c.N, c.K, False)


def dgrad_plan(c):
    if c.fp32:
        return "simt", None
    if c.tma and c.N % 4 == 0:
        return "tma", tma_plan(c.B, c.K, c.N, True, False, tma_ok(c.out_off, c.K))
    return "staged", staged_plan(c.B, c.K, c.N, False)


def wgrad_plan(c):
    if c.fp32:
        return "simt", None
    if c.tma and c.N % 4 == 0 and tma_ok(c.x_off, c.ldx):
        return "tma", tma_plan(c.N, c.K, c.B, True, True, tma_ok(c.out_off, c.K))
    return "staged", staged_plan(c.N, c.K, c.B, True)


def branches(c, drop=False):
    s = set()
    if c.ldx > c.K:
        s.add("x:padded")
    if c.op == "fwd":
        path, p = fwd_plan(c)
        s.add(f"fwd:{path}")
        if path == "tma":
            s |= _tma_labels("fwd", p, c.B, c.N, c.K, True, c.out_off, c.N)
        elif path == "staged":
            if p["n_tiles"] > 1:
                s.add("fwd:staged_n_tiles>1")
        if drop:
            s.add("drop:fused" if path == "tma" else "drop:kernel")
        return s
    if c.N == 1:
        if c.K <= GEMV_BWD_MAX:
            s.add("bwd1:gemv_bwd8" if c.K <= GEMV4_MAX else "bwd1:gemv_bwd16")
            if c.wants("dx") and c.dx_mask:
                s.add("bwd1:gemv_bwd_mask")
            if c.wants("dw") or c.wants("db"):
                s.add("bwd1:colsum_parts")
        else:
            if c.wants("dx"):
                s.add("bwd1:outer_rows_mask" if c.dx_mask else "bwd1:outer_rows")
            if c.wants("dw"):
                s.add("bwd1:colsum_dw")
            if c.wants("db"):
                s.add("bwd1:colsum_db")
        return s
    db_done = False
    if c.wants("dx"):
        path, p = dgrad_plan(c)
        s.add(f"dgrad:{path}")
        if path == "tma":
            s |= _tma_labels("dgrad", p, c.B, c.K, c.N, False, c.out_off, c.K)
            if c.presplit:
                s.add("dgrad:presplit")
            if c.dx_mask:
                m_tma = p["c_tma"] and tma_ok(c.x_off, c.ldx) and p["smem"] + M_STAGE_BYTES <= MASK_BUDGET
                s.add("dgrad:mask_tma" if m_tma else "dgrad:mask_thread")
        elif c.dx_mask:
            s.add("dgrad:mask_rows_kernel")
    if c.wants("dw"):
        path, p = wgrad_plan(c)
        s.add(f"wgrad:{path}")
        if path == "tma":
            if p["splits"] == 1:
                s.add("wgrad:splits1_c_tma" if p["c_tma"] else "wgrad:splits1_c_thread")
            else:
                s.add("wgrad:splitk")
                last = p["kb"] - (p["splits"] - 1) * p["kps"]
                if c.B % BK == 1 and last < p["kps"]:
                    s.add("wgrad:short_last_split_one_row")
            if p["n_tiles"] > 1 and p["splits"] > 1:
                s.add("wgrad:n_tiles>1_x_splits")
            if c.B % BK == BK - 1:
                s.add("wgrad:k%32==31")
            if c.wants("db"):
                s.add("db:converter+reduce2" if p["splits"] > 1 else "db:converter+reduce")
                db_done = True
        elif path == "staged" and p["splits"] > 1:
            s.add("wgrad:staged_splitk")
    if c.wants("db") and not db_done:
        s.add("db:colsum_kernel")
    return s


def _fwd(name, B, K, N, note="", **kw):
    return Case(name, "fwd", B, K, N, note=note, **kw)


def _bwd(name, B, K, N, note="", **kw):
    return Case(name, "bwd", B, K, N, note=note, **kw)


FWD_CASES = [
    _fwd("f_b1_k4", 1, 4, 300, "one row, K below one k-block"),
    _fwd("f_b129_k8", 129, 8, 200, "one row in the 2nd m-tile; 112-column tile, 16-column tail"),
    _fwd("f_two_tiles", 18944, 150, 300, "148*128 rows: every CTA takes two tiles", ldx=152),
    _fwd("f_149_tiles", 18945, 1, 16, "149 tiles of the narrowest width", ldx=4),
    _fwd("f_k33_n1100", 300, 33, 1100, "7 n-tiles, bias from global, K % 32 == 1", ldx=36),
    _fwd("f_e32", 513, 64, 1030, "per-thread 32-column epilogue, bias from global, cvec 2"),
    _fwd("f_e16", 999, 100, 75, "16-column epilogue, cvec 1"),
    _fwd("f_padded_y4", 777, 100, 300, "padded x; y 4 bytes off 16", ldx=108, out_off=1),
    _fwd("f_y8", 300, 64, 200, "y 8 bytes off 16", out_off=2),
    _fwd("f_bench_150", 65536, 150, 300, "benchmark layer 150 -> 300", ldx=152),
    _fwd("f_bench_300", 65536, 300, 200, "benchmark layer 300 -> 200"),
    _fwd("f_x_misaligned", 777, 100, 300, "x 4 bytes off 16: staged kernel", x_off=1),
    _fwd("f_staged_env", 300, 33, 1100, "RLCTR_GEMM_TMA=0: staged kernel, 5 n-tiles", tma=False),
    _fwd("f_staged_e16", 999, 100, 75, "RLCTR_GEMM_TMA=0", tma=False),
    _fwd("f_fp32_32", 1000, 150, 300, "RLCTR_MLP_FP32, 32x32 tiles", fp32=True),
    _fwd("f_fp32_64", 1024, 64, 1200, "RLCTR_MLP_FP32, 64x64 tiles", fp32=True),
    _fwd("f_gemv4", 1000, 152, 1, "out 1, aligned rows of 152"),
    _fwd("f_gemv_350", 1000, 350, 1, "out 1, in 350 (DCN at D = 10)"),
    _fwd("f_gemv_680", 1000, 680, 1, "out 1, in 680 (DCN at D = 32)"),
    _fwd("f_gemv_odd_ldx", 1000, 150, 1, "out 1, odd pitch", ldx=151),
]

BWD_CASES = [
    _bwd("g_777_600_300", 777, 600, 300, "4 n-tiles, TMA C and TMA mask", dx_mask=True),
    _bwd("g_777_600_300_nomask", 777, 600, 300, "", want="dx"),
    _bwd("g_777_presplit", 777, 600, 300, "weight images from the forward call", dx_mask=True, presplit=True, want="dx"),
    _bwd("g_1000_1100_64", 1000, 1100, 64, "7 n-tiles", dx_mask=True, want="dx,db"),
    _bwd("g_18945_36_300", 18945, 36, 300, "149 tiles; C store and mask per thread: shared memory is full",
         dx_mask=True, presplit=True, want="dx"),
    _bwd("g_mask_pitch", 777, 600, 300, "mask pitch 601: mask per thread; wgrad staged", ldx=601, dx_mask=True),
    _bwd("g_dx_off4", 777, 600, 300, "dx 4 bytes off 16: C per thread", out_off=1, dx_mask=True, want="dx"),
    _bwd("g_out75", 999, 100, 75, "out 75: staged + mask_rows_kernel, colsum db", dx_mask=True),
    _bwd("g_staged_env", 777, 600, 300, "RLCTR_GEMM_TMA=0", tma=False, dx_mask=True),
    _bwd("g_fp32", 1000, 150, 300, "RLCTR_MLP_FP32", fp32=True, dx_mask=True),
    _bwd("w_300_152_200", 300, 152, 200, "splits 1: dW through TMA, db from the colsum partial"),
    _bwd("w_dw_off8", 300, 152, 200, "splits 1, dW 8 bytes off 16: per-thread store", out_off=2, want="dw,db"),
    _bwd("w_2047_300_200", 2047, 300, 200, "8 splits, K % 32 == 31", want="dw,db"),
    _bwd("w_40001_36_304", 40001, 36, 304, "49 splits, the last of 3 k-blocks, the last holding one row", want="dw,db"),
    _bwd("w_1100_1024_1024", 1100, 1024, 1024, "7 n-tiles x 2 splits", want="dw,db"),
    _bwd("w_ldx_odd", 2047, 300, 200, "x pitch 301: staged split-K", ldx=301, want="dw,db"),
    _bwd("b_bench_150", 65536, 150, 300, "benchmark layer 150 -> 300", ldx=152, presplit=True),
    _bwd("b_bench_300", 65536, 300, 200, "benchmark layer 300 -> 200", dx_mask=True, presplit=True),
]
for _k in (150, 350, 680):
    BWD_CASES += [
        _bwd(f"o_{_k}_all", 1000, _k, 1, "out 1", ldx=_k + (2 if _k == 150 else 0)),
        _bwd(f"o_{_k}_all_mask", 1000, _k, 1, "out 1", dx_mask=True),
        _bwd(f"o_{_k}_dx", 1000, _k, 1, "out 1", want="dx"),
        _bwd(f"o_{_k}_dx_mask", 1000, _k, 1, "out 1", dx_mask=True, want="dx"),
        _bwd(f"o_{_k}_dw", 1000, _k, 1, "out 1", want="dw"),
        _bwd(f"o_{_k}_db", 1000, _k, 1, "out 1", want="db"),
    ]

# dropout: (case, counter) -- the fused epilogue of each kind and the elementwise kernel, at every counter edge
DROP_CASES = [
    _fwd("d_c_tma", 300, 64, 300, "fused, TMA C store"),
    _fwd("d_e32", 513, 64, 1030, "fused, per-thread 32-column chunks"),
    _fwd("d_e16", 999, 100, 75, "fused, 16-column chunks"),
    _fwd("d_kernel", 300, 64, 300, "dropout_kernel", tma=False),
    _fwd("d_kernel_75", 999, 100, 75, "dropout_kernel", tma=False),
]
SEED = 0x1234_5678_9ABC_DEF1


def cross_counter(N, row=5, col=40):
    """a counter just below 2^33 that puts element 2^33 (pair index 2^32) at (row, col): inside a 32- and a 16-column chunk"""
    return (1 << 33) - (row * N + col)


def counters(N):
    return {"ctr0": 0, "odd": 12345, "cross2^33": cross_counter(N), "above2^40": (1 << 40) + 3 * (1 << 33) + 6}


def chunk_starts(c):
    """first column of every epilogue chunk of the fused dropout (chunk width per column range)"""
    path, p = fwd_plan(c)
    out = []
    for nt in range(p["n_tiles"]):
        base, n_tile = nt * p["n_tile"], p["n_tile"]
        if p["c_tma"]:
            out += [(base + 32 * j, 32) for j in range(n_tile // 32)]
            if n_tile % 32:
                out.append((base + n_tile // 32 * 32, 16))
        else:
            w = 32 if n_tile % 32 == 0 else 16
            out += [(base + w * j, w) for j in range(n_tile // w)]
    return [(n0, w) for n0, w in out if n0 < c.N]


def drop_branches(c, ctr):
    """which formula the fused epilogue takes: the one-key fast path, the per-element path, the 2^32 pair crossing"""
    s = branches(c, drop=True)
    if ctr + c.B * c.N > (1 << 33):
        s.add("drop:pair_hi>0")
    if "drop:fused" not in s:
        return s
    m = np.arange(c.B, dtype=np.uint64)[:, None]
    for n0, w in chunk_starts(c):
        i0 = np.uint64(ctr) + m * np.uint64(c.N) + np.uint64(n0)
        cross = (i0 >> np.uint64(33)) != ((i0 + np.uint64(w - 1)) >> np.uint64(33))
        odd = (i0 & np.uint64(1)) == 1
        if odd.all():
            s.add("drop:slow_every_row")
        elif odd.any():
            s.add("drop:slow_odd_rows")
        if cross.any():
            s.add("drop:slow_pair_crossing")
        if (~odd & ~cross).any():
            s.add("drop:fast")
    return s


REQUIRED = {
    "fwd:tma", "fwd:staged", "fwd:simt32", "fwd:simt64", "fwd:gemv_rows4", "fwd:gemv_rows", "x:padded",
    "fwd:cta_second_tile", "fwd:n_tiles>1", "fwd:k<32", "fwd:k%32==1", "fwd:c_tma", "fwd:c_tma+tail16", "fwd:e32",
    "fwd:e16", "fwd:bias_smem", "fwd:bias_global", "fwd:cvec1", "fwd:cvec2", "fwd:staged_n_tiles>1",
    "dgrad:tma", "dgrad:staged", "dgrad:simt", "dgrad:c_tma", "dgrad:c_thread_smem", "dgrad:cvec1", "dgrad:mask_tma",
    "dgrad:mask_thread", "dgrad:mask_rows_kernel", "dgrad:presplit", "dgrad:cta_second_tile", "dgrad:n_tiles>1",
    "wgrad:tma", "wgrad:staged", "wgrad:simt", "wgrad:splits1_c_tma", "wgrad:splits1_c_thread", "wgrad:splitk",
    "wgrad:short_last_split_one_row", "wgrad:n_tiles>1_x_splits", "wgrad:k%32==31", "wgrad:staged_splitk",
    "db:converter+reduce", "db:converter+reduce2", "db:colsum_kernel",
    "bwd1:gemv_bwd8", "bwd1:gemv_bwd16", "bwd1:gemv_bwd_mask", "bwd1:colsum_parts", "bwd1:outer_rows",
    "bwd1:outer_rows_mask", "bwd1:colsum_dw", "bwd1:colsum_db",
    "drop:fused", "drop:kernel", "drop:fast", "drop:slow_every_row", "drop:slow_odd_rows", "drop:slow_pair_crossing",
    "drop:pair_hi>0",
}


def table():
    rows = []
    for c in FWD_CASES + BWD_CASES:
        rows.append((c.name, f"B {c.B} in {c.K} out {c.N}" + (f" ldx {c.ldx}" if c.ldx != c.K else ""),
                     " ".join(sorted(b for b in branches(c) if b != "x:padded"))))
    for c in DROP_CASES:
        labs = set()
        for ctr in counters(c.N).values():
            labs |= drop_branches(c, ctr)
        rows.append((c.name, f"B {c.B} in {c.K} out {c.N}", " ".join(sorted(b for b in labs if b.startswith("drop:")))))
    w0 = max(len(r[0]) for r in rows)
    w1 = max(len(r[1]) for r in rows)
    return "\n".join(f"    {a:<{w0}}  {b:<{w1}}  {t}" for a, b, t in rows)


# ---------------------------------------------------------------------------------------------------------------------------
# exact operand families
# ---------------------------------------------------------------------------------------------------------------------------
LO = 2.0 ** -13


def dyadic(rng, shape):
    """a + b * 2^-13, a in {-1, 0, 1}, b in {-3 .. 3}"""
    return (rng.integers(-1, 2, shape) + rng.integers(-3, 4, shape) * LO).astype(np.float32)


def small_int(rng, shape):
    return rng.integers(-1, 2, shape).astype(np.float32)


def dyadic_bias(rng, n):
    return (rng.integers(-4 * 8192, 4 * 8192 + 1, n) * LO).astype(np.float32)


def sparse(rng, a, density):
    return np.where(rng.random(a.shape) < density, a, np.float32(0)).astype(np.float32)


def frac_bits(a, device="cpu"):
    """least e with a * 2^e integral (e <= 40; operands here need at most 15)"""
    t = torch.as_tensor(np.ascontiguousarray(a), device=device).double()
    for e in range(41):
        u = t * 2.0 ** e
        if bool((u == u.floor()).all()):
            return e
    raise AssertionError("operand is not on a dyadic grid")


def exact_window(A, Bm, bias=None, device="cpu"):
    """(max over outputs of sum_k |A_mk Bm_nk| + |bias_n|, 2^(23 - e)) with 2^-e the grid of the products: the precondition of
    the exact families is first < second"""
    e = frac_bits(A, device) + frac_bits(Bm, device)
    if bias is not None:
        e = max(e, frac_bits(bias, device))
    s = torch.as_tensor(np.ascontiguousarray(A), device=device).double().abs() @ \
        torch.as_tensor(np.ascontiguousarray(Bm), device=device).double().abs().T
    if bias is not None:
        s = s + torch.as_tensor(bias, device=device).double().abs()
    return (float(s.max()) if s.numel() else 0.0), 2.0 ** (23 - e)


def fwd_operands(fam, B, K, N, seed):
    rng = np.random.default_rng(seed)
    if fam == "A":
        return dyadic(rng, (B, K)), small_int(rng, (N, K)), dyadic_bias(rng, N)
    if fam == "B":
        return small_int(rng, (B, K)), dyadic(rng, (N, K)), dyadic_bias(rng, N)
    return (rng.standard_normal((B, K)).astype(np.float32), (rng.standard_normal((N, K)) / np.sqrt(K)).astype(np.float32),
            rng.standard_normal(N).astype(np.float32))


def bwd_density(B, N):
    """dy sparse enough that every dgrad row sum and wgrad / db column sum stays far inside the window"""
    return min(1.0, 64.0 / N, 128.0 / B)


def bwd_operands(fam, B, K, N, seed):
    """(x [B, K], w [N, K], dy [B, N], y [B, N]): y is the saved layer output the ReLU backward masks with"""
    rng = np.random.default_rng(seed)
    y = rng.standard_normal((B, N)).astype(np.float32)
    if fam == "A":
        d = bwd_density(B, N)
        return small_int(rng, (B, K)), small_int(rng, (N, K)), sparse(rng, dyadic(rng, (B, N)), d), y
    if fam == "B":
        d = bwd_density(B, N)
        return dyadic(rng, (B, K)), dyadic(rng, (N, K)), sparse(rng, small_int(rng, (B, N)), d), y
    return (rng.standard_normal((B, K)).astype(np.float32), (rng.standard_normal((N, K)) / np.sqrt(K)).astype(np.float32),
            rng.standard_normal((B, N)).astype(np.float32), y)


def fwd_inputs(c, fam):
    return fwd_operands(fam, c.B, c.K, c.N, c.B * 7 + c.K * 3 + c.N)


def bwd_inputs(c, fam, relu):
    """x, w, dy, the saved output y, the dy the GEMMs see (after the in-place ReLU backward), gy_scale and dx_scale"""
    x, w, dy, y = bwd_operands(fam, c.B, c.K, c.N, c.B * 5 + c.K * 11 + c.N + relu)
    gy_scale = float(dropout_scale(0.2)) if relu else 1.0     # the tower's ReLU + dropout backward: 1 / (1 - p)
    dx_scale = float(dropout_scale(0.2)) if relu else 2.0
    dy_eff = np.where(y > 0, dy * np.float32(gy_scale), np.float32(0)).astype(np.float32) if relu else dy
    return x, w, dy, y, dy_eff, gy_scale, dx_scale


def bwd_windows(x, w, dy_eff, device="cpu"):
    """the exactness precondition of dgrad (rows of dy w), wgrad (columns of dy^T x) and db (column sums of dy)"""
    ones = np.ones((1, dy_eff.shape[0]), np.float32)
    return [exact_window(a, bm, None, device) for a, bm in ((dy_eff, w.T), (dy_eff.T, x.T), (dy_eff.T, ones))]


# ---------------------------------------------------------------------------------------------------------------------------
# the dropout mask of common.cuh (mix32 / dropout_key / dropout_bits / dropout_keep) in numpy
# ---------------------------------------------------------------------------------------------------------------------------
def mix32(x):
    x = np.asarray(x, np.uint32).copy()
    with np.errstate(over="ignore"):
        x ^= x >> np.uint32(16)
        x *= np.uint32(0x7FEB352D)
        x ^= x >> np.uint32(15)
        x *= np.uint32(0x846CA68B)
        x ^= x >> np.uint32(16)
    return x


def dropout_key(seed, pair_hi):
    s_lo, s_hi = np.uint32(seed & 0xFFFFFFFF), np.uint32(seed >> 32)
    return mix32(s_lo ^ mix32(s_hi ^ np.asarray(pair_hi, np.uint32) ^ np.uint32(0x9E3779B9)))


def dropout_bits(key, pair_lo):
    return mix32(np.asarray(pair_lo, np.uint32) ^ key)


def keep(seed, idx, thresh):
    """per-element formula (dropout_keep): idx uint64 element indices"""
    idx = np.asarray(idx, np.uint64)
    pair = idx >> np.uint64(1)
    h = dropout_bits(dropout_key(seed, (pair >> np.uint64(32)).astype(np.uint32)), (pair & np.uint64(0xFFFFFFFF)).astype(np.uint32))
    r = np.where((idx & np.uint64(1)) == 1, h >> np.uint32(16), h & np.uint32(0xFFFF))
    return r >= np.uint32(thresh)


def keep_chunk_fast(seed, i0, w, thresh):
    """the fused epilogue's fast path for one chunk of w columns starting at element i0 (even, no 2^32 pair crossing):
    one key for the chunk, one hash per pair"""
    assert i0 % 2 == 0 and (i0 >> 33) == ((i0 + w - 1) >> 33)
    p0 = i0 >> 1
    key = dropout_key(seed, np.uint32(p0 >> 32))
    h = dropout_bits(key, (np.uint32(p0 & 0xFFFFFFFF) + np.arange(w // 2, dtype=np.uint32)).astype(np.uint32))
    out = np.empty(w, bool)
    out[0::2] = (h & np.uint32(0xFFFF)) >= thresh
    out[1::2] = (h >> np.uint32(16)) >= thresh
    return out


def dropout_thresh(p):
    return int(min(max(float(np.float32(p)) * 65536.0, 0.0), 65535.0))


def dropout_scale(p):
    return np.float32(1.0) / (np.float32(1.0) - np.float32(p))


# ---------------------------------------------------------------------------------------------------------------------------
# GPU harness: guarded buffers, NaN workspace, immutability, determinism
# ---------------------------------------------------------------------------------------------------------------------------
SENT = 0x7FC0DEAD           # a quiet NaN with a payload no kernel writes
GUARD = 64                  # floats of sentinel before and after every buffer: 256 bytes, two 128-byte lines


@pytest.fixture(scope="module")
def lib():
    from rl_ctr_prediction_b200 import _lib
    return _lib.load()


def _L():
    from rl_ctr_prediction_b200 import _lib
    return _lib


class Guarded:
    """A flat fp32 view of n floats, `off` floats past a 256-byte boundary, inside sentinel NaN guards."""

    def __init__(self, n, off=0, fill=None):
        self.n, self.lo = n, GUARD + off
        self.base = torch.full((GUARD + off + n + GUARD,), SENT, dtype=torch.int32, device=DEV).view(torch.float32)
        assert self.base.data_ptr() % 256 == 0
        self.view = self.base[self.lo:self.lo + n]
        if fill is not None:
            self.view.copy_(torch.as_tensor(np.ascontiguousarray(fill).reshape(-1), device=DEV))

    @property
    def ptr(self):
        return self.view.data_ptr()

    def guards_ok(self):
        b = self.base.view(torch.int32)
        return bool((b[:self.lo] == SENT).all()) and bool((b[self.lo + self.n:] == SENT).all())


def matrix_buf(a, ld, extra_rows, off=0):
    """a [R, C] at pitch ld inside a guarded buffer; pad columns and `extra_rows` rows past R hold NaN"""
    R, Cn = a.shape
    full = np.full((R + extra_rows, ld), np.nan, np.float32)
    full[:R, :Cn] = a
    return Guarded(full.size, off, full)


def ws_buf(lib, B, K, N):
    nb = lib.rlctr_mlp_ws_bytes(B, K, N)
    assert nb == ws_layout(B, K, N)["total"], (nb, ws_layout(B, K, N))
    ws = torch.empty(nb // 4, dtype=torch.int32, device=DEV)
    return ws, nb


def nan_fill(ws, keep_images=None):
    """every word of the workspace to the sentinel, except [images, images + 2*wsplit) when keep_images = layout"""
    if keep_images is None:
        ws.fill_(SENT)
    else:
        a, b = keep_images["images"] // 4, (keep_images["images"] + 2 * keep_images["wsplit"]) // 4
        ws[:a].fill_(SENT)
        ws[b:].fill_(SENT)


def t64(a):
    return torch.as_tensor(np.ascontiguousarray(a), device=DEV).double()


def scaled(v32, mask, s):
    """np.float32(v) * np.float32(s) where mask, else 0 -- one fp32 multiply, as the kernels do"""
    return torch.where(mask, v32 * torch.tensor(float(np.float32(s)), dtype=torch.float32, device=DEV), torch.zeros_like(v32))


def check_precision(got, ref64, ref32, vs_sgemm=True):
    """family R: the close() bar of test_gpu_kernels.py (1e-5 of the output scale plus 1e-5 of the element) against fp64, and
    (vs_sgemm) within 16x of fp32 SGEMM's own error.  dW is exempt from the second bound: its k is the batch, and the tensor
    core's fp32 accumulator truncates instead of rounding, so over 65536 rows the 3xTF32 dW carries an error biased toward zero
    (1.3e-5 of the scale at 300 -> 200, 8.6e-6 at 150 -> 300 with the ReLU backward, measured on a B200) that is inside the bar
    but 18-30x cuBLAS's blocked sums"""
    scale = float(ref64.abs().max()) if ref64.numel() else 0.0
    diff = (got.double() - ref64).abs()
    assert bool((diff <= 1e-5 * scale + 1e-5 * ref64.abs()).all()), (float(diff.max()), scale)
    if vs_sgemm and ref64.numel():
        err, err32 = float(diff.max()), float((ref32.double() - ref64).abs().max())
        assert err <= max(16 * err32, 2e-6 * scale), (err, err32, scale)


def fwd_call(lib, c, xg, wg, bg, y, flags, p, rng_state, ws, nb):
    L = _L()
    return lib.rlctr_linear_fwd(xg.ptr, c.ldx, wg.ptr, bg.ptr, y.ptr, c.B, c.K, c.N, flags, p,
                                rng_state.data_ptr() if rng_state is not None else None, ws.data_ptr(), nb, L.stream())


def run_fwd(lib, c, fam, relu, monkeypatch, drop_p=0.0, ctr=0):
    """one forward case: returns (y as fp32 tensor [B, N], fp64 pre-dropout reference, the operands)"""
    L = _L()
    monkeypatch.setenv("RLCTR_GEMM_TMA", "1" if c.tma else "0")
    x, w, b = fwd_inputs(c, fam)
    if fam != "R":
        s, lim = exact_window(x, w, b, DEV)
        assert s < lim, (c.name, s, lim)
    xg = matrix_buf(x, c.ldx, 3, c.x_off)
    wg, bg = Guarded(w.size, 0, w), Guarded(c.N, 0, b)
    inputs = [(g, g.base.view(torch.int32).clone()) for g in (xg, wg, bg)]
    ws, nb = ws_buf(lib, c.B, c.K, c.N)
    flags = (L.RLCTR_MLP_RELU if relu else 0) | (L.RLCTR_MLP_FP32 if c.fp32 else 0) | (L.RLCTR_MLP_DROPOUT if drop_p else 0)
    st = torch.tensor([SEED, ctr], dtype=torch.int64, device=DEV) if drop_p else None
    outs = []
    for _ in range(2):
        nan_fill(ws)
        y = Guarded(c.B * c.N, c.out_off)
        assert fwd_call(lib, c, xg, wg, bg, y, flags, drop_p, st, ws, nb) == 0
        torch.cuda.synchronize()
        assert y.guards_ok(), c.name
        outs.append(y)
    for g, before in inputs:
        assert torch.equal(g.base.view(torch.int32), before), c.name
    assert torch.equal(outs[0].view.view(torch.int32), outs[1].view.view(torch.int32)), "second run differs"
    if drop_p:
        assert int(st[1]) == ctr                               # the forward call does not move the counter
    ref = t64(x) @ t64(w).T + t64(b)
    if relu:
        ref = ref.clamp_min(0)
    return outs[0].view.view(c.B, c.N), ref, (x, w, b)


FWD_IDS = [c.name for c in FWD_CASES]


@pytest.mark.parametrize("fam", ["A", "B", "R"])
@pytest.mark.parametrize("relu", [0, 1])
@pytest.mark.parametrize("case", FWD_CASES, ids=FWD_IDS)
def test_linear_fwd_edges(lib, case, relu, fam, monkeypatch):
    y, ref, (x, w, b) = run_fwd(lib, case, fam, relu, monkeypatch)
    if fam == "R":
        ref32 = torch.as_tensor(x, device=DEV) @ torch.as_tensor(w, device=DEV).T + torch.as_tensor(b, device=DEV)
        check_precision(y, ref, ref32.clamp_min(0) if relu else ref32)
    else:
        assert torch.equal(y, ref.float()), (case.name, float((y.double() - ref).abs().max()))


DROP_PARAMS = [(c, k, p) for c in DROP_CASES for k in counters(c.N) for p in (0.5, 0.2)]


@pytest.mark.parametrize("fam", ["A", "B"])
@pytest.mark.parametrize("case,ctr_name,p", DROP_PARAMS, ids=[f"{c.name}-{k}-p{p}" for c, k, p in DROP_PARAMS])
def test_linear_fwd_dropout_bits(lib, case, ctr_name, p, fam, monkeypatch):
    """y = keep(seed, counter + m*N + n) ? relu(x w^T + b) * fp32(1/(1-p)) : 0, bit for bit against the numpy port of the hash"""
    ctr = counters(case.N)[ctr_name]
    y, ref, _ = run_fwd(lib, case, fam, 1, monkeypatch, drop_p=p, ctr=ctr)
    idx = np.uint64(ctr) + np.arange(case.B * case.N, dtype=np.uint64)
    k = torch.as_tensor(keep(SEED, idx, dropout_thresh(p)).reshape(case.B, case.N), device=DEV)
    want = scaled(ref.float(), k, dropout_scale(p))
    assert torch.equal(y, want), (case.name, ctr_name, int((y != want).sum()))
    # kept and dropped both occur (the reference is not vacuous), and the fraction is about 1 - p
    frac = float(k.float().mean())
    assert abs(frac - (1 - p)) < 0.02, frac


BWD_IDS = [c.name for c in BWD_CASES]


@pytest.mark.parametrize("fam", ["A", "B", "R"])
@pytest.mark.parametrize("relu", [0, 1])
@pytest.mark.parametrize("case", BWD_CASES, ids=BWD_IDS)
def test_linear_bwd_edges(lib, case, relu, fam, monkeypatch):
    L = _L()
    c = case
    monkeypatch.setenv("RLCTR_GEMM_TMA", "1" if c.tma else "0")
    x, w, dy, yv, dy_eff, gy_scale, dx_scale = bwd_inputs(c, fam, relu)
    if fam != "R":
        for s, lim in bwd_windows(x, w, dy_eff, DEV):
            assert s < lim, (c.name, s, lim)
    xg = matrix_buf(x, c.ldx, 3, c.x_off)
    wg = Guarded(w.size, 0, w)
    yg = Guarded(yv.size, 0, yv)
    frozen = [(g, g.base.view(torch.int32).clone()) for g in (xg, wg, yg)]
    ws, nb = ws_buf(lib, c.B, c.K, c.N)
    lay = ws_layout(c.B, c.K, c.N)
    flags = ((L.RLCTR_MLP_RELU if relu else 0) | (L.RLCTR_MLP_DX_MASK if c.dx_mask else 0) | (L.RLCTR_MLP_FP32 if c.fp32 else 0) |
             (L.RLCTR_MLP_W_PRESPLIT if c.presplit else 0))
    runs = []
    for _ in range(2):
        gyg = matrix_buf(dy, c.N, 2)                           # rows past B hold NaN; the ReLU backward rewrites dy in place
        nan_fill(ws)
        if c.presplit:                                         # the layer's forward call leaves (W_hi, W_lo) in the workspace
            yf = Guarded(c.B * c.N)
            bz = Guarded(c.N, 0, np.zeros(c.N, np.float32))
            assert fwd_call(lib, c, xg, wg, bz, yf, 0, 0.0, None, ws, nb) == 0
            nan_fill(ws, keep_images=lay)
        outs = {k: (Guarded(n, c.out_off) if c.wants(k) else None)
                for k, n in (("dx", c.B * c.K), ("dw", c.N * c.K), ("db", c.N))}
        ptr = lambda g: g.ptr if g is not None else None
        assert lib.rlctr_linear_bwd(xg.ptr, c.ldx, wg.ptr, yg.ptr if relu else None, gyg.ptr, ptr(outs["dx"]), ptr(outs["dw"]),
                                    ptr(outs["db"]), c.B, c.K, c.N, flags, gy_scale, dx_scale, ws.data_ptr(), nb,
                                    L.stream()) == 0
        torch.cuda.synchronize()
        for k, g in outs.items():
            if g is not None:
                assert g.guards_ok(), (c.name, k)
        assert gyg.guards_ok()
        runs.append((outs, gyg))
    for g, before in frozen:
        assert torch.equal(g.base.view(torch.int32), before), c.name
    outs, gyg = runs[0]
    for k in outs:
        if outs[k] is not None:
            assert torch.equal(outs[k].view.view(torch.int32), runs[1][0][k].view.view(torch.int32)), (c.name, k, "second run")
    # dy: unchanged, or masked and scaled in place; the NaN rows past B untouched
    gy_t = gyg.view.view(c.B + 2, c.N)
    assert torch.isnan(gy_t[c.B:]).all()
    assert torch.equal(gy_t[:c.B], torch.as_tensor(dy_eff, device=DEV)), c.name
    d64, x64, w64 = t64(dy_eff), t64(x), t64(w)
    refs = {"dx": d64 @ w64, "dw": d64.T @ x64, "db": d64.sum(0)}
    if c.dx_mask:
        maskx = torch.as_tensor(x > 0, device=DEV)
    for k, g in outs.items():
        if g is None:
            continue
        got = g.view.view(*refs[k].shape)
        if fam == "R":
            d32, x32, w32 = (torch.as_tensor(a, device=DEV) for a in (dy_eff, x, w))
            r32 = {"dx": d32 @ w32, "dw": d32.T @ x32, "db": d32.sum(0)}[k]
            ref = refs[k]
            if k == "dx" and c.dx_mask:
                ref, r32 = ref * maskx * dx_scale, r32 * maskx * dx_scale
            check_precision(got, ref, r32, vs_sgemm=k != "dw")
        else:
            want = refs[k].float()
            if k == "dx" and c.dx_mask:
                want = scaled(want, maskx, dx_scale)
            assert torch.equal(got, want), (c.name, k, float((got.double() - want.double()).abs().max()))


if __name__ == "__main__":
    print(table())
    sys.exit(0)
