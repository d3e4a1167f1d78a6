"""CUDA-graph train step of every get_model name at D = 10, 16 and 32 (B = 65536, F = 15, N = 10M, uniform ids; FFM at D = 32
on N = 2M: its 484-float rows with Adam state take 5.8 KB per id), plus the per-call time of the kernels the latent size
selects, their algorithmic bytes / FLOP, and the share of a device-to-device copy measured in the same run:

    python scratch/latent_dims_bench.py [--steps 20] [--out profiles/latent_dims_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rl_ctr_prediction_b200 import _lib, graphs, optim, pretrain_main as PM  # noqa: E402

B, F, N = 65536, 15, 10_000_000
NAMES = ["LR", "FM", "FFM", "W&D", "DeepFM", "FNN", "IPNN", "OPNN", "DCN", "AFM"]
DIMS = [10, 16, 32]
KERNELS = ("rlctr_embed_fwd", "rlctr_ffm_fwd", "rlctr_rows_adam", "rlctr_afm_fwd", "rlctr_afm_bwd", "rlctr_cross_fwd",
           "rlctr_cross_bwd")


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else torch.cuda.get_device_name(0)
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0)


def copy_peak_gbs(dev):
    """Device-to-device copy of 2 GiB (read + write bytes over time): the attainable HBM rate the shares are taken against."""
    a = torch.empty(1 << 29, dtype=torch.float32, device=dev)
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    return 2 * a.numel() * 4 * 10 / (e0.elapsed_time(e1) * 1e-3) / 1e9


def algorithmic(key, meta, D, rs):
    """(bytes, flop) one call needs at the least: rows read once, outputs written once, FLOP of the interaction."""
    fd, P, n = F * D, F * (F - 1) // 2, B * F
    if key.startswith("rlctr_embed_fwd"):
        return n * rs * 4 + B * (rs + fd + 1) * 4, 0
    if key.startswith("rlctr_ffm_fwd"):
        return n * rs * 4 + n * rs * 4 + B * 4, B * P * 2 * D
    if key.startswith("rlctr_rows_adam"):
        return n * rs * 4 + n * 3 * rs * 4 * 2, n * rs * 20            # gradient rows in; (p, m, v) read + written per occurrence
    if key.startswith("rlctr_afm_fwd"):
        return B * fd * 4 + B * 4, B * P * (2 * D * D + 5 * D)
    if key.startswith("rlctr_afm_bwd"):
        return 2 * B * fd * 4 + B * 4, B * P * (6 * D * D + 12 * D)
    if key.startswith("rlctr_cross_fwd"):
        return 2 * B * fd * 4, B * 5 * 4 * fd
    if key.startswith("rlctr_cross_bwd"):
        return 3 * B * fd * 4, B * 5 * 8 * fd
    return 0, 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    ap.add_argument("--names", default=",".join(NAMES))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    info = gpu_info()
    peak = copy_peak_gbs(dev)
    print(info, f"copy peak {peak:.0f} GB/s", flush=True)
    lossf = torch.nn.BCELoss()
    results = []
    for D in DIMS:
        for name in args.names.split(","):
            n_rows = 2_000_000 if (name == "FFM" and D == 32) else N
            torch.manual_seed(1)
            m = PM.get_model(name, n_rows, F, D)
            with torch.no_grad():
                m.table.mul_(0.1)
            m = m.to(dev).train()
            opt = optim.Adam(m.parameters(), lr=1e-3, weight_decay=1e-5)
            gen = torch.Generator(device=dev).manual_seed(D)
            data = [(torch.randint(0, n_rows, (B, F), generator=gen, device=dev),
                     (torch.rand(B, generator=gen, device=dev) < 0.05).to(torch.int64)) for _ in range(args.steps + 4)]
            # per-call kernel times: eager steps under the KernelTimer (a run of its own, before the graph is captured)
            timer = _lib.KernelTimer()
            _lib.set_timer(timer)
            for x, y in data[:4]:
                graphs.eager_step(m, opt, lossf, x, y)
            _lib.set_timer(None)
            rs = m._geom.row_stride
            kern = {}
            for key, (count, ms, _) in timer.summary().items():
                if not key.startswith(KERNELS):
                    continue
                nbytes, flop = algorithmic(key, None, D, rs)
                kern[key] = {"ms": round(ms, 4), "alg_MB": round(nbytes / 1e6, 1), "alg_GFLOP": round(flop / 1e9, 2),
                             "GB_s": round(nbytes / (ms * 1e-3) / 1e9, 0), "copy_peak_share": round(nbytes / (ms * 1e-3) / 1e9 / peak, 3),
                             "TFLOP_s": round(flop / (ms * 1e-3) / 1e12, 2)}
            gstep = graphs.GraphedTrainStep([(m, opt)], lossf, eager_steps=2)
            for x, y in data[:4]:
                gstep(x, y)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for x, y in data[4:]:
                gstep(x, y)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / args.steps
            r = {"model": name, "D": D, "N": n_rows, "row_floats": rs, "step_ms": round(ms, 4),
                 "samples_per_s_M": round(B / (ms * 1e-3) / 1e6, 2), "kernels": kern}
            print(json.dumps(r), flush=True)
            results.append(r)
            del gstep, m, opt, data
            torch.cuda.empty_cache()
    out = {"gpu": info, "copy_peak_GB_s": round(peak, 0), "B": B, "F": F, "ids": "uniform", "results": results}
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
