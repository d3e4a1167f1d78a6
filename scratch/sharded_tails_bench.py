"""Row-sharded co-located groups with tail members: CUDA-graph step of sharded.ShardedGroup at the C2 shape (B = 65536 per GPU,
N = 10M, F = 15, D = 10, uniform ids), one rank per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node G --master-addr 127.0.0.1 --master-port 29519 \\
        scratch/sharded_tails_bench.py [--steps 20] [--rounds 3] [--out profiles/sharded_tails_bench.json]

G = 1 (a one-rank NCCL group, symmetric memory as plain tensors): colocated.ColocatedCTR on the same batches beside it, alternated.
G > 1: an in-process A/B of the merged push (one rlctr_push_rows_routed_multi call) against one rlctr_push_rows_routed per member into
per-member buffers, on the same routing workspace, timed with CUDA events.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rl_ctr_prediction_b200 import _lib, colocated, graphs, optim, pretrain_main as PM, sharded  # noqa: E402

B, F, D, N = 65536, 15, 10, 10_000_000
COMBOS = {"LR+FM+FNN": ("LR", "FM", "FNN"), "DeepFM+IPNN": ("DeepFM", "IPNN"), "AFM+LR+DCN": ("AFM", "LR", "DCN")}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else torch.cuda.get_device_name(0)
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0)


def make_group(names, dev):
    ms = []
    for i, n in enumerate(names):
        torch.manual_seed(1 + i)
        m = PM.get_model(n, N, F, D)
        with torch.no_grad():
            m.table.mul_(0.1)
        ms.append(m.to(dev).train())
    return colocated.colocate(ms)


def time_steps(step, data):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for x, y in data:
        step(x, y)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / len(data)


def push_ab(sg, x, reps=50):
    """Merged push vs one push per tail member, same routing workspace (ms per call, median of three windows each)."""
    lib, G, rank, st = _lib.load(), sg.world, sg.rank, _lib.stream()
    n = x.numel()
    view = sharded.routed_view_pos(x, sg.feature_nums, sg.group)
    tails, pitch = sg._tail_sources()
    srcs = [torch.randn(n, w, device=x.device) for _, _, w in tails]
    merged = sg._exchange(B, F)["recv"][1]
    per = []
    for _, _, w in tails:
        pm = sharded.PeerMemory(G * view["cap"] * w, torch.float32, x.device, sg.group)
        per.append((pm, (C.c_void_p * 8)(*[int(p) for p in pm.ptrs])))
    sp = (C.c_void_p * len(srcs))(*[s.data_ptr() for s in srcs])
    wd = (C.c_int32 * len(srcs))(*[w for _, _, w in tails])

    def merged_call():
        _lib.check(lib.rlctr_push_rows_routed_multi(view["route_ws"].data_ptr(), n, G, rank, view["cap"], sp, wd, len(srcs), merged,
                                                    st), "push multi")

    def separate_calls():
        for s, (_, ptrs), (_, _, w) in zip(srcs, per, tails):
            _lib.check(lib.rlctr_push_rows_routed(view["route_ws"].data_ptr(), n, G, rank, view["cap"], s.data_ptr(), w, ptrs, st),
                       "push")

    out = {"merged": [], "separate": []}
    for r in range(6):
        for k, fn in (("merged", merged_call), ("separate", separate_calls))[::(1 if r % 2 == 0 else -1)]:
            sg.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            out[k].append(e0.elapsed_time(e1) / reps)
    sg.barrier()
    return {k: round(sorted(v)[len(v) // 2], 4) for k, v in out.items()} | {"sources": len(srcs), "pitch": pitch}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    G, rank = dist.get_world_size(), dist.get_rank()
    gen = torch.Generator(device=dev).manual_seed(1 + rank)
    per = N // F
    data = []
    for _ in range(args.steps + 4):
        x = torch.randint(0, per, (B, F), generator=gen, device=dev, dtype=torch.int64) + torch.arange(F, device=dev) * per
        data.append((x, (torch.rand(B, generator=gen, device=dev) < 0.05).to(torch.int64)))
    results = []
    for label, names in COMBOS.items():
        cg = make_group(names, dev)
        sg = sharded.ShardedGroup.from_group(cg)
        arms = {"sharded_group": (sg, graphs.GraphedTrainStep([(sg, optim.Adam(sg.parameters(), lr=1e-3, weight_decay=1e-5))]))}
        if G == 1:
            arms["colocated"] = (cg, graphs.GraphedTrainStep([(cg, optim.Adam(cg.parameters(), lr=1e-3, weight_decay=1e-5))]))
        else:
            del cg
        for _, step in arms.values():
            for x, y in data[:4]:                         # two eager steps, the capture, one replay
                step(x, y)
        ms = {k: [] for k in arms}
        for r in range(args.rounds):
            order = list(arms) if r % 2 == 0 else list(arms)[::-1]
            for k in order:
                ms[k].append(time_steps(arms[k][1], data[4:]))
        row = {"combo": label, "world": G, "B_per_gpu": B, "N": N, "F": F, "D": D, "gpu": gpu_info(), "steps": args.steps,
               "rounds": args.rounds}
        for k in arms:
            assert arms[k][1].graph is not None
            med = sorted(ms[k])[len(ms[k]) // 2]
            row[k] = {"ms_per_step_rounds": [round(v, 4) for v in ms[k]], "ms_per_step_median": round(med, 4),
                      "samples_per_s_per_gpu": round(B / med * 1e3)}
        if G > 1 and sg._tail_sources()[0]:
            row["push_ms"] = push_ab(sg, data[0][0])
        else:
            row["push_ms"] = "not measured (one GPU: no routed push at world 1)"
        if rank == 0:
            print(json.dumps(row), flush=True)
        results.append(row)
        del arms, sg
        torch.cuda.empty_cache()
    if args.out and rank == 0:
        with open(args.out, "w") as fh:
            json.dump(results, fh, indent=1)
    torch.cuda.synchronize()
    sys.stdout.flush()
    os._exit(0)


if __name__ == "__main__":
    main()
