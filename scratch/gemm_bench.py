"""Times rlctr_linear_fwd / rlctr_linear_bwd on the DeepFM tower shapes, TMA kernel vs software-staged kernel."""
import os, sys, json
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rl_ctr_prediction_b200 import _lib

lib = _lib.load()
dev = torch.device("cuda:0")
B = int(os.environ.get("GB", 65536))
FAST = os.environ.get("GEMM_BENCH_FAST", "0") != "0"      # the TMA kernel on the two tower shapes only


def timeit(fn, n=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3


def run(K, N, ld):
    x = torch.randn(B, ld, device=dev)
    w = torch.randn(N, K, device=dev) / K ** 0.5
    b = torch.randn(N, device=dev)
    y = torch.empty(B, N, device=dev)
    gy = torch.randn(B, N, device=dev)
    dx = torch.empty(B, K, device=dev)
    dw = torch.empty(N, K, device=dev)
    db = torch.empty(N, device=dev)
    wsb = lib.rlctr_mlp_ws_bytes(B, K, N)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    st = _lib.stream()
    out = {}
    for mode in (("1",) if FAST else ("1", "0")):
        os.environ["RLCTR_GEMM_TMA"] = mode
        f = lambda: _lib.check(lib.rlctr_linear_fwd(x.data_ptr(), ld, w.data_ptr(), b.data_ptr(), y.data_ptr(), B, K, N, 1, 0.0, None, ws.data_ptr(), wsb, st), "fwd")
        d = lambda: _lib.check(lib.rlctr_linear_bwd(x.data_ptr(), ld, w.data_ptr(), None, gy.data_ptr(), dx.data_ptr(), None, None, B, K, N, 0, 1.0, 1.0, ws.data_ptr(), wsb, st), "dgrad")
        g = lambda: _lib.check(lib.rlctr_linear_bwd(x.data_ptr(), ld, w.data_ptr(), None, gy.data_ptr(), None, dw.data_ptr(), None, B, K, N, 0, 1.0, 1.0, ws.data_ptr(), wsb, st), "wgrad")
        tag = "tma" if mode == "1" else "staged"
        fl = 2.0 * B * K * N
        dm = lambda: _lib.check(lib.rlctr_linear_bwd(x.data_ptr(), ld, w.data_ptr(), None, gy.data_ptr(), dx.data_ptr(), None, None, B, K, N, _lib.RLCTR_MLP_DX_MASK, 1.0, 2.0, ws.data_ptr(), wsb, st), "dgrad_mask")
        for name, fn in (("fwd", f), ("dgrad", d), ("dgrad_mask", dm), ("wgrad", g)):
            us = timeit(fn)
            out[f"{tag}.{name}"] = {"us": round(us, 1), "fp32_TFLOPs": round(fl / us / 1e6, 1)}
    # cuBLAS on the same shapes (verdict r1: is 76-116 fp32-equivalent TFLOP/s good?): SGEMM (allow_tf32 = False: what the reference's
    # nn.Linear runs on a GPU) and cuBLAS' own 1xTF32 (1e-3 error: fails the 1e-5 parity bar, shown as the tensor-core ceiling)
    xk = x[:, :K].contiguous()
    fl = 2.0 * B * K * N
    for tag, tf32 in (() if FAST else (("cublas_sgemm", False), ("cublas_tf32", True))):
        torch.backends.cuda.matmul.allow_tf32 = tf32
        yy = torch.empty(B, N, device=dev)
        for name, fn in (("fwd", lambda: torch.addmm(b, xk, w.t(), out=yy)), ("dgrad", lambda: torch.mm(gy, w, out=dx)),
                         ("wgrad", lambda: torch.mm(gy.t(), xk, out=dw))):
            us = timeit(fn)
            out[f"{tag}.{name}"] = {"us": round(us, 1), "fp32_TFLOPs": round(fl / us / 1e6, 1)}
    torch.backends.cuda.matmul.allow_tf32 = False
    ref = x[:, :K].double() @ w.double().T + b.double()
    os.environ["RLCTR_GEMM_TMA"] = "1"
    _lib.check(lib.rlctr_linear_fwd(x.data_ptr(), ld, w.data_ptr(), b.data_ptr(), y.data_ptr(), B, K, N, 0, 0.0, None, ws.data_ptr(), wsb, st), "fwd")
    out["max_rel_err_fwd"] = float(((y.double() - ref).abs().max() / ref.abs().max()).item())
    return out


for K, N, ld in ((150, 300, 152), (300, 200, 300), (256, 304, 256), (1024, 1024, 1024))[:2 if FAST else 4]:
    print(json.dumps({"B": B, "K": K, "N": N, "ld": ld, **run(K, N, ld)}), flush=True)
