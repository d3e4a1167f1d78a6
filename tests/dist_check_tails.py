#!/usr/bin/env python
"""1-vs-G equivalence of the row-sharded tail models on real GPUs (run under torchrun, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29518 tests/dist_check_tails.py

ShardedCTR for WideAndDeep / FNN / InnerPNN / OuterPNN / DCN / AFM, and ShardedGroup for [DeepFM, InnerPNN], [WideAndDeep, DCN] and
[AFM, LR, DCN], trained on G ranks x B/G, against the single-GPU model (colocated.ColocatedCTR for the groups) on the global batch.
Dropout is off (towers in eval(), AFM dropout_p = 0): with it on, each rank draws its own masks.  Tolerances: dist_check.within.
Prints one JSON line per model; exits non-zero on a mismatch."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from dist_check import within  # noqa: E402
from rl_ctr_prediction_b200 import colocated, optim, pretrain_main as PM, sharded  # noqa: E402


def _no_dropout(m):
    m.eval()
    if hasattr(m, "dropout_p"):
        m.dropout_p = 0.0
    return m


def _dense_errs(a, b, prefix=""):
    """Max relative error of every dense parameter of a (sharded) against b (single GPU), keyed like dist_check's tower weights."""
    pb = dict(b.named_parameters())
    errs = {}
    for k, p in a.named_parameters():
        if k == "table":
            continue
        scale = max(pb[k].abs().max().item(), 1e-12)
        errs[f"mlp.{prefix}{k}"] = ((p - pb[k]).abs().max() / scale).item()
    return errs


def _batch(rng, N, F, B, dev):
    x = torch.as_tensor(rng.integers(0, N, size=(B, F))).to(dev)
    y = torch.as_tensor((rng.random(B) < 0.3).astype(np.int64)).to(dev)
    return x, y


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    N, F, D, B, STEPS = 5003, 15, 10, 256 * world, 4
    lo, hi = rank * (B // world), (rank + 1) * (B // world)
    ok = True
    for name in ("W&D", "FNN", "IPNN", "OPNN", "DCN", "AFM"):
        torch.manual_seed(7)
        single = PM.get_model(name, N, F, D)
        with torch.no_grad():
            single.table.mul_(0.1)
        _no_dropout(single.to(dev))
        m = sharded.ShardedCTR.from_model(single)
        m.eval()
        opt_s = optim.Adam(single.parameters(), lr=1e-3, weight_decay=1e-5)
        opt_m = optim.Adam(m.parameters(), lr=1e-3, weight_decay=1e-5)
        rng = np.random.default_rng(11)
        lossf = torch.nn.BCELoss()
        for s in range(STEPS):
            x, y = _batch(rng, N, F, B, dev)
            tl = lossf(single(x), y.unsqueeze(1).float())
            single.zero_grad()
            tl.backward()
            opt_s.step()
            m.train_step(x[lo:hi].contiguous(), y[lo:hi].contiguous(), opt_m)
        single.flush()
        full = m.gather_table()
        scale = single.table.data.abs().max().item()
        errs = {"table": (full - single.table.data).abs().max().item() / scale}
        errs.update(_dense_errs(m.dense, single))
        good = within(errs)
        ok = ok and good
        if rank == 0:
            print(json.dumps({"model": name, "world": world, "ok": good, "max_rel_err_vs_single_gpu": errs}), flush=True)
    for names in (("DeepFM", "IPNN"), ("W&D", "DCN"), ("AFM", "LR", "DCN")):
        torch.manual_seed(9)
        members = [PM.get_model(n, N, F, D) for n in names]
        for mm in members:
            with torch.no_grad():
                mm.table.mul_(0.1)
            _no_dropout(mm.to(dev))
        cg = colocated.colocate(members)
        sg = sharded.ShardedGroup.from_group(cg)
        opt_s = optim.Adam(cg.parameters(), lr=1e-3, weight_decay=1e-5)
        opt_m = optim.Adam(sg.parameters(), lr=1e-3, weight_decay=1e-5)
        rng = np.random.default_rng(13)
        for s in range(STEPS):
            x, y = _batch(rng, N, F, B, dev)
            cg.train_step(x, y, opt_s)
            sg.train_step(x[lo:hi].contiguous(), y[lo:hi].contiguous(), opt_m)
        cg.flush()
        full = sg.gather_table()
        rs = cg._geom.row_stride
        scale = cg.table.data[:, :rs].abs().max().item()
        errs = {"table": (full - cg.table.data)[:, :rs].abs().max().item() / scale,
                "exp_avg_sq": ((full - cg.table.data)[:, 64:64 + rs].abs().max() / cg.table.data[:, 64:64 + rs].abs().max()).item()}
        for i, (a, b) in enumerate(zip(sg.members, cg.members)):
            errs.update(_dense_errs(a, b, prefix=f"{i}."))
        good = within(errs)
        ok = ok and good
        if rank == 0:
            print(json.dumps({"model": "group(" + "+".join(names) + ")", "world": world, "ok": good,
                              "max_rel_err_vs_single_gpu": errs}), flush=True)
    if rank == 0:
        print("ok" if ok else "MISMATCH", flush=True)
    # every rank has printed / compared; leave without tearing the symmetric-memory mappings down collectively
    torch.cuda.synchronize()
    sys.stdout.flush()
    os._exit(0 if ok else 1)


if __name__ == "__main__":
    main()
