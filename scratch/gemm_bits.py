"""SHA-256 of the raw outputs of the tower GEMM entry points on seeded inputs, one line per (shape, call), so that two builds can
be compared byte for byte:  python scratch/gemm_bits.py OUT_FILE  (then `cmp` the files of two trees).

Calls: rlctr_linear_fwd with ReLU + dropout, dgrad, masked dgrad (mask rows TMA can address, and at pitch K + 1, which it cannot),
and wgrad with db.  Shapes: the scratch/gemm_bench.py tower shapes at B = 65536 (their wgrads are split-K), a smaller split-K
wgrad, a single-split wgrad, and an output pitch TMA cannot store to."""
import hashlib
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rl_ctr_prediction_b200 import _lib

RELU, DROPOUT, DX_MASK = 1, 2, 4
SHAPES = [(65536, 150, 300), (65536, 300, 200), (65536, 256, 304), (65536, 1024, 1024),   # (B, K = in_dim, N = out_dim)
          (1000, 150, 300), (200, 300, 200), (999, 100, 75)]


def main(out):
    lines = []
    lib = _lib.load()
    dev = torch.device("cuda:0")
    st = _lib.stream()
    ptr = _lib.ptr
    for B, K, N in SHAPES:
        g = torch.Generator().manual_seed(B * 7919 + K * 31 + N)
        ld = (K + 3) // 4 * 4
        x = torch.zeros(B, ld)
        x[:, :K] = torch.randn(B, K, generator=g)
        w = torch.randn(N, K, generator=g) / K ** 0.5
        b = torch.randn(N, generator=g)
        gy = torch.randn(B, N, generator=g)
        xm = torch.where(torch.rand(B, K, generator=g) < 0.4, 0.0, x[:, :K].abs())          # layer-below output: 0 where dropped
        x, w, b, gy = x.to(dev), w.to(dev), b.to(dev), gy.to(dev)
        xm_tma = torch.zeros(B, ld, device=dev)
        xm_tma[:, :K] = xm.to(dev)
        xm_odd = torch.zeros(B, K + 1, device=dev)
        xm_odd[:, :K] = xm.to(dev)
        wsb = lib.rlctr_mlp_ws_bytes(B, K, N)
        ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
        rng = torch.tensor([1234567, 0], dtype=torch.int64, device=dev)
        y = torch.empty(B, N, device=dev)
        dx = torch.empty(B, K, device=dev)
        dxm = torch.empty(B, K, device=dev)
        dxo = torch.empty(B, K, device=dev)
        dw = torch.empty(N, K, device=dev)
        db = torch.empty(N, device=dev)
        s = 1.0 / (1.0 - 0.2)
        _lib.check(lib.rlctr_linear_fwd(ptr(x), ld, ptr(w), ptr(b), ptr(y), B, K, N, RELU | DROPOUT, 0.2, ptr(rng), ptr(ws), wsb, st),
                   "fwd")
        _lib.check(lib.rlctr_linear_bwd(ptr(x), ld, ptr(w), None, ptr(gy), ptr(dx), None, None, B, K, N, 0, 1.0, 1.0, ptr(ws), wsb,
                                        st), "dgrad")
        _lib.check(lib.rlctr_linear_bwd(ptr(xm_tma), ld, ptr(w), None, ptr(gy), ptr(dxm), None, None, B, K, N, DX_MASK, 1.0, s,
                                        ptr(ws), wsb, st), "dgrad_mask")
        _lib.check(lib.rlctr_linear_bwd(ptr(xm_odd), K + 1, ptr(w), None, ptr(gy), ptr(dxo), None, None, B, K, N, DX_MASK, 1.0, s,
                                        ptr(ws), wsb, st), "dgrad_mask_pitch")
        _lib.check(lib.rlctr_linear_bwd(ptr(x), ld, ptr(w), None, ptr(gy), None, ptr(dw), ptr(db), B, K, N, 0, 1.0, 1.0, ptr(ws),
                                        wsb, st), "wgrad")
        torch.cuda.synchronize()
        for name, t in (("fwd", y), ("dgrad", dx), ("dgrad_mask", dxm), ("dgrad_mask_pitch", dxo), ("wgrad_dw", dw),
                        ("wgrad_db", db)):
            lines.append(f"{B}x{K}x{N} {name} {hashlib.sha256(t.cpu().numpy().tobytes()).hexdigest()}")
            print(lines[-1], flush=True)
        assert torch.equal(dxm, dxo), (B, K, N)          # the mask through TMA == the mask read per thread
    with open(out, "w") as fh:
        fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main(sys.argv[1])
