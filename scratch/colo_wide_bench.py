"""Wide co-located records against stand-alone tables: the CUDA-graph train step of each group of DESIGN §6b ("Wide records") as one
joint record (colocate(..., max_lines=4)) and as one table per model in one captured step, B = 65536, F = 15, N = 10M, uniform ids,
the two alternated three times in one process; plus the per-call time of the row-side kernels (eager steps under _lib.KernelTimer):

    python scratch/colo_wide_bench.py [--steps 20] [--out profiles/colo_wide_bench.json]
"""
import argparse
import copy
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rl_ctr_prediction_b200 import _lib, colocated, graphs, optim, pretrain_main as PM  # noqa: E402

B, F, N = 65536, 15, 10_000_000
SHAPES = [(("LR", "FM", "DeepFM"), 16), (("LR", "FM", "DeepFM"), 32), (("FM", "FNN", "DeepFM"), 10)]
ROW_KERNELS = ("rlctr_group_fwd", "rlctr_embed_fwd", "rlctr_rows_catchup", "rlctr_group_rows_adam", "rlctr_rows_adam")


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else torch.cuda.get_device_name(0)
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0)


def build(names, D, dev):
    torch.manual_seed(1)
    torch.set_default_device(dev)
    try:
        ms = [PM.get_model(n, N, F, D) for n in names]
    finally:
        torch.set_default_device(None)
    for m in ms:
        with torch.no_grad():
            m.table.mul_(0.1)
        m.to(dev).train()
    return ms


def row_kernels(step_fn, data):
    timer = _lib.KernelTimer()
    _lib.set_timer(timer)
    for x, y in data:
        step_fn(x, y)
    _lib.set_timer(None)
    return {k: {"calls": c, "ms": round(ms, 4)} for k, (c, ms, _) in timer.summary().items() if k.startswith(ROW_KERNELS)}


def timed(gstep, data):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for x, y in data:
        gstep(x, y)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / len(data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    info = gpu_info()
    print(info, flush=True)
    lossf = torch.nn.BCELoss()
    results = []
    for names, D in SHAPES:
        sep = build(names, D, dev)
        grp = [copy.deepcopy(m) for m in sep]
        group = colocated.colocate(grp, max_lines=4)
        opts = [optim.Adam(m.parameters(), lr=1e-3, weight_decay=1e-5) for m in sep]
        gopt = optim.Adam(group.parameters(), lr=1e-3, weight_decay=1e-5)
        gen = torch.Generator(device=dev).manual_seed(D)
        data = [(torch.randint(0, N, (B, F), generator=gen, device=dev),
                 (torch.rand(B, generator=gen, device=dev) < 0.05).to(torch.int64)) for _ in range(args.steps + 4)]
        k_sep = row_kernels(lambda x, y: [graphs.eager_step(m, o, lossf, x, y) for m, o in zip(sep, opts)], data[:4])
        k_grp = row_kernels(lambda x, y: group.train_step(x, y, gopt), data[:4])
        s_sep = graphs.GraphedTrainStep(list(zip(sep, opts)), lossf)
        s_grp = graphs.GraphedTrainStep([(group, gopt)], lossf)
        for x, y in data[:4]:
            s_sep(x, y)
            s_grp(x, y)
        t_sep, t_grp = [], []
        for _ in range(3):                                   # alternated in one process: separate, joint, separate, joint ...
            t_sep.append(timed(s_sep, data[4:]))
            t_grp.append(timed(s_grp, data[4:]))
        g = group._geom
        r = {"members": list(names), "D": D, "N": N, "B": B, "joint_row_floats": g.row_stride, "record_pitch_floats": g.row_pitch,
             "separate_step_ms": [round(v, 4) for v in t_sep], "joint_step_ms": [round(v, 4) for v in t_grp],
             "separate_row_kernels": k_sep, "joint_row_kernels": k_grp}
        print(json.dumps(r), flush=True)
        results.append(r)
        del s_sep, s_grp, group, gopt, opts, sep, grp, data
        torch.cuda.empty_cache()
    out = {"gpu": info, "B": B, "F": F, "N": N, "ids": "uniform", "results": results}
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
