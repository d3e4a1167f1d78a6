"""Timings for optimizer checkpoints (writes one JSON line).

    python scratch/optim_state_bench.py eager     # eager FM step (B = 65536, N = 10M, Adam wd 1e-5): ms per step
    python scratch/optim_state_bench.py ckpt      # C2 group (co-located LR + FM + DeepFM, N = 10M): state_dict / load_state_dict

``eager`` runs from any tree of this project (it uses no API the optimizer checkpoints added), so the same command times the
parent's step against this one's.  Every time ends in a device synchronise; the card's name and power limit are read in the same
run."""
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.getcwd())


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def _batches(N, F, B, k, dev):
    g = torch.Generator(device=dev).manual_seed(0)
    return [(torch.randint(0, N, (B, F), device=dev, generator=g), torch.randint(0, 2, (B, 1), device=dev, generator=g))
            for _ in range(k)]


def eager(N=10_000_000, F=15, D=10, B=65536, steps=200, warmup=20):
    from rl_ctr_prediction_b200 import graphs, optim, pretrain_main as PM
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    m = PM.get_model("FM", N, F, D).to(dev)
    opt = optim.Adam(m.parameters(), lr=1e-3, weight_decay=1e-5)
    lossf = torch.nn.BCELoss()
    bs = _batches(N, F, B, 8, dev)
    for i in range(warmup):
        graphs.eager_step(m, opt, lossf, *bs[i % 8])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(steps):
        graphs.eager_step(m, opt, lossf, *bs[i % 8])
    torch.cuda.synchronize()
    return {"what": "eager FM step", "tree": os.getcwd(), "ms_per_step": (time.perf_counter() - t0) * 1e3 / steps,
            "steps": steps, "card": _card()}


def ckpt(N=10_000_000, F=15, D=10, B=65536, reps=5):
    import io
    from rl_ctr_prediction_b200 import colocated, optim, pretrain_main as PM
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    g = colocated.colocate([PM.get_model(n, N, F, D).to(dev) for n in ("LR", "FM", "DeepFM")])
    opt = optim.Adam(g.parameters(), lr=1e-3, weight_decay=1e-5)
    for x, y in _batches(N, F, B, 4, dev):
        g.train_step(x, y, opt)
    out = {"what": "C2 group optimizer checkpoint", "N": N, "card": _card()}
    times = {"state_dict": [], "state_dict_to_cpu": [], "load_state_dict_from_cpu": []}
    for _ in range(reps):
        x, y = _batches(N, F, B, 1, dev)[0]
        g.train_step(x, y, opt)                                 # rows behind again: the export includes the flush
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sd = opt.state_dict()
        torch.cuda.synchronize()
        times["state_dict"].append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        cpu = {"state": {i: {k: (v.cpu() if isinstance(v, torch.Tensor) else v) for k, v in e.items()}
                         for i, e in sd["state"].items()}, "param_groups": sd["param_groups"]}
        times["state_dict_to_cpu"].append(time.perf_counter() - t0)
        del sd
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        opt.load_state_dict(cpu)
        torch.cuda.synchronize()
        times["load_state_dict_from_cpu"].append(time.perf_counter() - t0)
    out.update({k: {"median_ms": sorted(v)[len(v) // 2] * 1e3, "all_ms": [t * 1e3 for t in v]} for k, v in times.items()})
    buf = io.BytesIO()
    torch.save(cpu, buf)
    out["checkpoint_bytes"] = buf.tell()
    return out


if __name__ == "__main__":
    print(json.dumps({"eager": eager, "ckpt": ckpt}[sys.argv[1]]()))
