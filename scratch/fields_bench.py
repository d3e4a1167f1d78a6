"""CUDA-graph train step of every get_model name at F = 15, 24, 39 and 64 with D = 8 (B = 65536, N = 10M uniform ids; FFM on
N = 2M: its F*D + 1 floats a row with Adam state), plus the per-call time of the pair dots (InnerPNN) and the FFM forward
through _lib.KernelTimer, and the card's name, power limit and max SM clock read in the same run:

    python scratch/fields_bench.py [--steps 20] [--out profiles/fields_bench.json]

AFM serves F <= 23 only and is timed at F = 15; DCN at F = 64 runs at D = 8 (F*D = 512, its limit); FFM at F = 64 at D = 7
(rows of 512 floats are the update's limit)."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rl_ctr_prediction_b200 import _lib, graphs, optim, pretrain_main as PM  # noqa: E402

B, N, D0 = 65536, 10_000_000, 8
FIELDS = [15, 24, 39, 64]
NAMES = ["LR", "FM", "FFM", "W&D", "DeepFM", "FNN", "IPNN", "OPNN", "DCN", "AFM"]
KERNELS = ("rlctr_pairdots_fwd", "rlctr_pairdots_bwd", "rlctr_ffm_fwd")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    ap.add_argument("--names", default=",".join(NAMES))
    ap.add_argument("--fields", default=",".join(map(str, FIELDS)))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    info = gpu_info()
    print(info, flush=True)
    lossf = torch.nn.BCELoss()
    results = []
    for F in map(int, args.fields.split(",")):
        for name in args.names.split(","):
            if name == "AFM" and F > 23:
                continue
            D = 7 if (name == "FFM" and F == 64) else D0
            n_rows = 2_000_000 if name == "FFM" else N
            torch.manual_seed(1)
            m = PM.get_model(name, n_rows, F, D)
            with torch.no_grad():
                m.table.mul_(0.1)
            m = m.to(dev).train()
            opt = optim.Adam(m.parameters(), lr=1e-3, weight_decay=1e-5)
            gen = torch.Generator(device=dev).manual_seed(F)
            data = [(torch.randint(0, n_rows, (B, F), generator=gen, device=dev),
                     (torch.rand(B, generator=gen, device=dev) < 0.05).to(torch.int64)) for _ in range(args.steps + 4)]
            timer = _lib.KernelTimer()
            _lib.set_timer(timer)
            for x, y in data[:4]:
                graphs.eager_step(m, opt, lossf, x, y)
            _lib.set_timer(None)
            kern = {key: {"calls": count, "ms": round(ms, 4)} for key, (count, ms, _) in timer.summary().items()
                    if key.startswith(KERNELS)}
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
            r = {"model": name, "F": F, "D": D, "N": n_rows, "row_floats": m._geom.row_stride, "step_ms": round(ms, 4),
                 "samples_per_s_M": round(B / (ms * 1e-3) / 1e6, 2), "kernels": kern}
            print(json.dumps(r), flush=True)
            results.append(r)
            del gstep, m, opt, data
            torch.cuda.empty_cache()
    out = {"gpu": info, "B": B, "ids": "uniform", "results": results}
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
