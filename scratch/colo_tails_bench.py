"""Co-located groups with a tail member against the same models trained stand-alone, A/B in one process on one GPU.

C2 shape: B = 65536, N = 10M, F = 15, D = 10, uniform ids.  For [LR, FM, FNN] and [DeepFM, InnerPNN]: the CUDA-graph step
(graphs.GraphedTrainStep) of the group and of the stand-alone models, alternated over several rounds so that both arms see the
same clocks and neighbours; then three eager steps of each arm under _lib.KernelTimer for the per-entry-point times.

    python scratch/colo_tails_bench.py [--steps 20] [--rounds 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rl_ctr_prediction_b200 import _lib, colocated, graphs, optim, pretrain_main as PM  # noqa: E402

B, F, D, N = 65536, 15, 10, 10_000_000
COMBOS = {"LR+FM+FNN": ("LR", "FM", "FNN"), "DeepFM+IPNN": ("DeepFM", "IPNN")}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else torch.cuda.get_device_name(0)
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0)


def make_models(names, dev):
    ms = []
    for i, n in enumerate(names):
        torch.manual_seed(1 + i)
        m = PM.get_model(n, N, F, D)
        with torch.no_grad():
            m.table.mul_(0.1)
        ms.append(m.to(dev).train())
    return ms


def build_arm(names, grouped, dev):
    ms = make_models(names, dev)
    if grouped:
        g = colocated.colocate(ms)
        pairs = [(g, optim.Adam(g.parameters(), lr=1e-3, weight_decay=1e-5))]
    else:
        pairs = [(m, optim.Adam(m.parameters(), lr=1e-3, weight_decay=1e-5)) for m in ms]
    return pairs, graphs.GraphedTrainStep(pairs, torch.nn.BCELoss())


def time_steps(step, data):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for x, y in data:
        step(x, y)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / len(data)


def kernel_times(pairs, data):
    t = _lib.KernelTimer()
    _lib.set_timer(t)
    try:
        for x, y in data:
            for m, opt in pairs:
                graphs.eager_step(m, opt, torch.nn.BCELoss(), x, y)
    finally:
        _lib.set_timer(None)
    return {k: round(v[1] * 1e3, 1) for k, v in sorted(t.summary().items())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    gen = torch.Generator(device=dev).manual_seed(1)
    per = N // F
    data = []
    for _ in range(args.steps + 4):
        x = torch.randint(0, per, (B, F), generator=gen, device=dev, dtype=torch.int64) + torch.arange(F, device=dev) * per
        data.append((x, (torch.rand(B, generator=gen, device=dev) < 0.05).to(torch.int64)))
    results = []
    for label, names in COMBOS.items():
        arms = {"group": build_arm(names, True, dev), "separate": build_arm(names, False, dev)}
        for _, step in arms.values():
            for x, y in data[:4]:                         # two eager steps, the capture, one replay
                step(x, y)
        ms = {k: [] for k in arms}
        for r in range(args.rounds):
            order = list(arms) if r % 2 == 0 else list(arms)[::-1]
            for k in order:
                ms[k].append(time_steps(arms[k][1], data[4:]))
        row = {"combo": label, "B": B, "N": N, "F": F, "D": D, "gpu": gpu_info(), "steps": args.steps, "rounds": args.rounds}
        for k in arms:
            assert arms[k][1].graph is not None
            best = sorted(ms[k])[len(ms[k]) // 2]
            row[k] = {"ms_per_step_rounds": [round(v, 4) for v in ms[k]], "ms_per_step_median": round(best, 4),
                      "samples_per_s": round(B / best * 1e3)}
        row["speedup_group_over_separate"] = round(row["separate"]["ms_per_step_median"] / row["group"]["ms_per_step_median"], 4)
        for k, (pairs, _) in arms.items():
            row[k]["kernel_us"] = kernel_times(pairs, data[:3])
        print(json.dumps(row), flush=True)
        results.append(row)
        del arms
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(results, fh, indent=1)


if __name__ == "__main__":
    main()
