"""optim.Adagrad against optim.Adam on the C2 workload: LR + FM + DeepFM co-located (one record per id), graphed step,
B = 65536, N = 10M rows, uniform ids over per-field ranges, D = 10.

Three optimizer settings alternate in one process on one group: Adam wd 1e-5 (the benchmark's), Adagrad wd 1e-5, Adagrad
wd 0.  Per setting: ms per graphed step (CUDA events over windows of replays, best and median window), then an eager pass
under _lib.KernelTimer for the per-call times of the row update and catch-up, and one timed flush of the whole table.
The card name and its power limit are read in the same run.

    python scratch/adagrad_bench.py --out profiles/adagrad_bench.json
"""
import argparse
import json
import statistics
import subprocess

import torch

from rl_ctr_prediction_b200 import _lib, colocated, graphs, optim, p_model

F, D = 15, 10


def batch(gen, B, N, dev):
    per = N // F
    x = torch.randint(0, per, (B, F), generator=gen, device=dev, dtype=torch.int64) + torch.arange(F, device=dev) * per
    y = (torch.rand(B, generator=gen, device=dev) < 0.05).to(torch.int64)
    return x, y


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


SETTINGS = {
    "adam_wd1e-5": lambda ps: optim.Adam(ps, lr=1e-3, weight_decay=1e-5),
    "adagrad_wd1e-5": lambda ps: optim.Adagrad(ps, lr=1e-2, weight_decay=1e-5),
    "adagrad_wd0": lambda ps: optim.Adagrad(ps, lr=1e-2),
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--steps", type=int, default=20, help="graph replays per timed window")
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=2, help="times the three settings are alternated")
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    B, N = args.batch, args.rows
    members = [p_model.LR(N, device=dev), p_model.FM(N, D, device=dev), p_model.DeepFM(N, F, D, device=dev)]
    with torch.no_grad():
        for m in members:
            m.table.mul_(0.1)
            m.train()
    group = colocated.colocate(members)
    del members
    torch.cuda.empty_cache()
    group.train()
    gen = torch.Generator(device=dev).manual_seed(0)
    batches = [batch(gen, B, N, dev) for _ in range(8)]
    res = {k: {"step_ms_windows": [], "calls": {}} for k in SETTINGS}
    for rnd in range(args.rounds):
        for name, make in SETTINGS.items():
            opt = make(group.parameters())                       # flushes what the previous optimizer owes, fresh state
            step = graphs.GraphedTrainStep([(group, opt)], torch.nn.BCELoss())
            for i in range(4):                                   # eager warm-up steps, capture, first replays
                step(*batches[i % len(batches)])
            torch.cuda.synchronize()
            for _ in range(args.windows):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for i in range(args.steps):
                    step(*batches[i % len(batches)])
                e1.record()
                torch.cuda.synchronize()
                res[name]["step_ms_windows"].append(e0.elapsed_time(e1) / args.steps)
            if rnd == args.rounds - 1:                           # per-call times: eager steps under the kernel timer, then a flush
                timer = _lib.KernelTimer()
                _lib.set_timer(timer)
                lossf = torch.nn.BCELoss()
                for i in range(10):
                    graphs.eager_step(group, opt, lossf, *batches[i % len(batches)])
                group.flush()
                summ = timer.summary()
                _lib.set_timer(None)
                res[name]["calls"] = {k: {"launches": n, "mean_ms": ms} for k, (n, ms, _) in summ.items()
                                      if any(s in k for s in ("rows_adam", "rows_adagrad", "catchup", "flush"))}
            del step
            torch.cuda.synchronize()
    for name, r in res.items():
        w = r["step_ms_windows"]
        r["step_ms_best"], r["step_ms_median"] = min(w), statistics.median(w)
    out = {"workload": f"C2: LR+FM+DeepFM co-located, graphed, B={B}, N={N}, D={D}, uniform ids",
           "card": card(), "settings": {"adam_wd1e-5": "optim.Adam(lr=1e-3, weight_decay=1e-5)",
                                        "adagrad_wd1e-5": "optim.Adagrad(lr=1e-2, weight_decay=1e-5)",
                                        "adagrad_wd0": "optim.Adagrad(lr=1e-2)"},
           "results": res}
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps({k: (round(v["step_ms_best"], 4), round(v["step_ms_median"], 4)) for k, v in res.items()}))


if __name__ == "__main__":
    main()
