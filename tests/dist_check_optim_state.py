#!/usr/bin/env python
"""Resume of row-sharded training at the same world size (run under torchrun, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29519 tests/dist_check_optim_state.py

For ShardedCTR (LR, FM, FFM, DeepFM) and ShardedGroup (LR + FM + DeepFM), with optim.Adam (wd 1e-5) and optim.Adagrad
(wd 1e-4): an uninterrupted run of K + M steps against a run that saves model and optimizer after K steps (torch.save to a
buffer, torch.load to the CPU) into a fresh sharded model and optimizer and trains M more.  The resumed run must equal the
uninterrupted one bit for bit (losses, gathered tables, optimizer state).  The gathered optimizer state must match a
single-GPU run on the concatenated batches within dist_check.py's bounds.  Prints one JSON line per case; exits non-zero on a
mismatch."""
import io
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rl_ctr_prediction_b200 import colocated, optim, pretrain_main as PM, sharded  # noqa: E402

SETTINGS = {"Adam": dict(lr=1e-3, weight_decay=1e-5), "Adagrad": dict(lr=1e-2, weight_decay=1e-4)}


def _save(model, opt):
    buf = io.BytesIO()
    torch.save({"model": model.state_dict(), "opt": opt.state_dict()}, buf)
    buf.seek(0)
    return torch.load(buf, map_location="cpu", weights_only=False)


def _single(name, N, F, D, dev, seed):
    torch.manual_seed(seed)
    m = PM.get_model(name, N, F, D)
    with torch.no_grad():
        m.table.mul_(0.1)
    return m.to(dev).eval()


def _tables(sd):
    return [e for e in sd["state"].values() if "geometry" in e]


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    N, F, D, B, K, M = 5003, 15, 10, 256 * world, 3, 3
    rng = np.random.default_rng(11)
    batches = [(torch.as_tensor(rng.integers(0, N, size=(B, F))).to(dev), torch.as_tensor((rng.random(B) < 0.3).astype(np.int64)).to(dev))
               for _ in range(K + M)]
    lo, hi = rank * (B // world), (rank + 1) * (B // world)
    local_batches = [(x[lo:hi].contiguous(), y[lo:hi].contiguous()) for x, y in batches]
    lossf = torch.nn.BCELoss()
    ok = True
    cases = [(n, c) for n in ("LR", "FM", "FFM", "DeepFM", "group") for c in SETTINGS]
    for name, cls in cases:
        make_opt = lambda m: getattr(optim, cls)(m.parameters(), **SETTINGS[cls])
        if name == "group":
            def make(seed):
                ms = [_single(n, N, F, D, dev, seed + i) for i, n in enumerate(("LR", "FM", "DeepFM"))]
                return colocated.colocate(ms)
            shard = lambda seed: sharded.ShardedGroup.from_group(make(seed))
            step = lambda m, o, x, y: m.train_step(x, y, o).cpu().tolist()
        else:
            make = lambda seed: _single(name, N, F, D, dev, seed)
            shard = lambda seed: sharded.ShardedCTR.from_model(make(seed))
            step = lambda m, o, x, y: float(m.train_step(x, y, o))
        a = shard(7)
        oa = make_opt(a)
        la = [step(a, oa, x, y) for x, y in local_batches]
        b = shard(7)
        ob = make_opt(b)
        lb = [step(b, ob, x, y) for x, y in local_batches[:K]]
        ck = _save(b, ob)
        c = shard(99)
        oc = make_opt(c)
        c.load_state_dict(ck["model"])
        oc.load_state_dict(ck["opt"])
        lb += [step(c, oc, x, y) for x, y in local_batches[K:]]
        sa, sc = oa.state_dict(), oc.state_dict()
        exact = la == lb and torch.equal(a.gather_table(), c.gather_table()) and all(
            all(torch.equal(u[k], v[k]) if isinstance(u[k], torch.Tensor) else u[k] == v[k] for k in u)
            for u, v in zip(_tables(sa), _tables(sc)))
        # the gathered state against the single-GPU run on the global batches
        single = make(7)
        os_ = make_opt(single)
        for x, y in batches:
            if name == "group":
                single.train_step(x, y, os_)
            else:
                from rl_ctr_prediction_b200 import graphs
                graphs.eager_step(single, os_, lossf, x, y)
        errs = {}
        for u, v in zip(_tables(sc), _tables(os_.state_dict())):
            for k in u:
                if isinstance(u[k], torch.Tensor):
                    errs[k] = ((u[k] - v[k]).abs().max() / v[k].abs().max().clamp_min(1e-30)).item()
        good = exact and all(e <= 2e-5 for e in errs.values())
        ok = ok and good
        if rank == 0:
            print(json.dumps({"model": name, "optimizer": cls, "world": world, "ok": good, "resume_bit_exact": exact,
                              "max_rel_err_state_vs_single_gpu": errs}))
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
