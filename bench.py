#!/usr/bin/env python
"""Benchmark of the hot path (BASELINE.json metric: train samples/sec + HBM roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]

Workload (SURVEY section 8d, config C2 == BASELINE.json configs[1]): one STEP = one training step of LR,
FM and DeepFM (forward, BCE loss, backward, Adam lr=1e-3 wd=1e-5 with the reference's dense-Adam
numerics) on ONE batch of B=65536 samples x F=15 fields, latent D=10, N=10,000,000 rows per table,
ids uniform over disjoint per-field ranges (tables >> L2, ~95% unique rows per batch), labels ~5% CTR.
value = B * steps / time: whole-job samples/s, inputs resident in HBM.  The lazy-exact optimizer's
flush (the pass that makes every untouched row equal to the reference's dense-Adam state) runs once
at the end INSIDE the timed region, so the tables at the end are the reference's tables.

e2e = the same steps through the drop-in API (model(x); BCELoss; zero_grad; backward; optimizer.step();
loss.item()) with each batch copied from pinned host memory inside the timed region.

--impl reference: the reference's own CPU implementation of the same step on all host threads: the reference's
modules themselves when its tree is importable (RLCTR_REF_PATH, /root/reference or baseline/_ref; `kind: "reference"`),
else oracle/torch_port.py (the same stock ATen CPU kernels the reference's modules call, dense torch.optim.Adam;
`kind: "port"`).  Under torchrun its global batch is batch x N, the B200 arm's global batch.

Beside the headline the line carries `configs` (the other BASELINE.json configurations: C1 FM B=4096 N=1e6, C3 REINFORCE
fused into the step, C4 FFM + DeepFM, C5 the src/all_main step at batch 1M), `steady_state` (median of several windows
without the end-of-run flush, the flush timed apart) and `gpu_eager_baseline` (stock PyTorch eager on the same B200:
the reference's loop body with dense torch.optim.Adam, BASELINE.md section 1).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

F_FIELDS = 15
MODELS = ("LR", "FM", "DeepFM")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dims", type=int, default=10)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cpu-steps", type=int, default=3)
    ap.add_argument("--no-graph", action="store_true", help="time the eager step instead of the CUDA-graph replay")
    ap.add_argument("--no-fork", action="store_true", help="capture the models of the step one after another (no parallel graph branches)")
    ap.add_argument("--no-colocate", action="store_true", help="single GPU: keep LR / FM / DeepFM in three separate tables instead "
                    "of one co-located record per id (rl_ctr_prediction_b200/colocated.py)")
    ap.add_argument("--profile-steps", type=int, default=10, help="steps of the eager per-kernel timing pass")
    ap.add_argument("--configs", default="C1,C3,C4,C5", help="other BASELINE.json configurations to time after the headline")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--no-eager-gpu", action="store_true", help="skip the stock-PyTorch-on-B200 baseline")
    ap.add_argument("--windows", type=int, default=5, help="steady-state windows of 20 steps after the headline region")
    ap.add_argument("--dump-outputs", metavar="DIR", help="one GPU: after the timed steps, write what the last one handed its "
                    "caller (every model's loss and its parameters after the flush) as DIR/<name>.npy")
    return ap.parse_args()


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def tensor_peak():
    """Dense TF32 tensor peak: half the bf16 rate (tcgen05 kind::tf32 has K = 8 per MMA where kind::f16 has 16)."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        return float(d["bf16_tflops_sustained"]) / 2.0, "measured bf16_tflops_sustained / 2 (MEASURED_PEAKS.json; tf32 = half the bf16 rate)"
    return 1400.0 / 2.0, "fallback 1.4 PFLOP/s sustained bf16 / 2 (B200_PROFILING.md)"


# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture of this round
NCU_TRAFFIC = {      # profiles/r2f_ncu_top_kernels.md (co-located step) / r2_ncu_top_kernels.md (three tables); B=65536, N=10M, D=10
    "rlctr_group_fwd[train]": 129.3e6 + 24.0e6, "rlctr_group_rows_adam": 443.0e6 + 232.7e6,
    "rlctr_rows_catchup[group]": 363.4e6 + 205.4e6,
    "rlctr_rows_adam[FM]": 247.7e6 + 139.0e6, "rlctr_rows_adam[DeepFM]": 297.2e6 + 141.5e6,
    "rlctr_rows_adam[LR]": 95.2e6 + 14.9e6,
    "rlctr_rows_catchup[FM]": 238.9e6 + 122.4e6, "rlctr_rows_catchup[DeepFM]": 238.9e6 + 122.7e6,
    "rlctr_rows_catchup[LR]": 91.1e6 + 12.1e6,
    "rlctr_embed_fwd[FM]": 68.3e6 + 3.7e6, "rlctr_embed_fwd[DeepFM]": 69.8e6 + 8.5e6, "rlctr_embed_fwd[LR]": 96.7e6 + 4.6e6,
    # the tower's calls, summed over their kernels (same capture): forward = 150->300, 300->200 GEMMs (+ the 200->1 GEMV, not captured);
    # backward = gemv_bwd + layer-2 dgrad, wgrad + layer-1 dgrad, wgrad
    "rlctr_linear_fwd": (40.3e6 + 23.8e6) + (79.2e6 + 20.3e6),
    "rlctr_linear_bwd": (52.7e6 + 7.5e6) + (131.7e6 + 45.0e6) + (131.2e6 + 5.1e6) + (79.1e6 + 4.2e6) + (118.7e6 + 4.1e6),
}


def make_batch(gen, B, N, device):
    """uniform ids over disjoint per-field ranges of N/F rows (SURVEY C2); ~5% positive labels."""
    per = N // F_FIELDS
    x = torch.randint(0, per, (B, F_FIELDS), generator=gen, device=device, dtype=torch.int64)
    x += torch.arange(F_FIELDS, device=device, dtype=torch.int64) * per
    y = (torch.rand(B, generator=gen, device=device) < 0.05).to(torch.int64)
    return x, y


def alg_bytes(key, m):
    """ALGORITHMIC bytes of one launch (DESIGN.md 'Kernels'; SURVEY section 8d): logical row sizes
    4*(D+1), int64 ids, each distinct row's Adam state read and written once.  U = expected number of
    distinct ids of a uniform batch."""
    name = key.split("[")[0]
    if name == "rlctr_sort_ids":
        return 16.0 * m["n"]                                   # read int64 ids, write u32 key + u32 slot
    if name == "rlctr_adam_flush":
        return m["n_rows"] * (24.0 * m["rs"] + 8.0)
    if name in ("rlctr_linear_fwd", "rlctr_linear_bwd"):
        return 0.0                                             # tensor-bound: reported in FLOP/s (gemm_flops)
    if name == "rlctr_bucket_by_owner":
        return 28.0 * m["n"]                                   # read int64 id; write int64 local row, int64 pos, u32 slot
    if name == "rlctr_gather_rows":
        return m["n"] * (8.0 + 8.0 * m["rs"])                  # id + row read + row write
    if "B" not in m:
        return 0.0
    B, F, N = m["B"], m["F"], m["n_rows"]
    logical = (m["dim"] + (1 if m["lin"] else 0)) if m["rs"] > 1 else 1
    n = B * F
    per = N / F
    U = F * per * (1.0 - (1.0 - 1.0 / per) ** B)
    if name in ("rlctr_group_fwd", "rlctr_group_rows_adam"):   # co-located record: `logical` = the members' parameters of one id
        M = len(m["members"])
        tower = sum(d for nm, d in m["members"] if nm in ("DeepFM", "WideAndDeep"))
        if name == "rlctr_group_fwd":
            train = "infer" not in key
            return float(B * (F * 8 + F * 4 * logical + 4 * M) + (B * 4 * logical if train else 0) + n * tower * 4)
        return float(U * (24 * logical + 8) + n * 8 + B * 4 * M + B * 4 * logical + n * tower * 4)
    if name == "rlctr_rows_lookup":                            # owner-side lookup: record read once, stage + gathered written
        return float(U * (24 * logical + 4) + n * (8 + 4 * logical))
    if name == "rlctr_embed_fwd":
        b = B * ((0 if m.get("streamed") else F * 8) + F * 4 * logical + 4)
        if m.get("sums"):
            b += B * 4 * logical
        if m.get("rows"):
            b += n * m["dim"] * 4
        return float(b)
    if name == "rlctr_rows_grad_dense":
        return float(n * (4 * logical * 2 + 8) + B * 4 * (1 + logical))
    if name == "rlctr_rows_adam":
        if m["model"].startswith("Sharded"):                   # owner side: n = rows received, gradients staged
            return float(U * 24 * logical + n * (8 + 4 * logical) + (U * 8 if m.get("stamp") else 0))
        b = U * 24 * logical + n * 8 + B * 4
        if m["model"] in ("FM", "DeepFM"):
            b += B * 4 * logical                               # saved column sums
        if m.get("extra"):
            b += n * m["dim"] * 4                              # tower input gradient
        if m.get("staged"):
            b += n * 4 * logical
        if m.get("stamp"):
            b += U * 8
        return float(b)
    if name == "rlctr_rows_catchup":
        # every distinct row that was NOT touched in the previous step is stale (uniform ids: a fraction U / N was): its record is
        # read, replayed and written back -- 24 * logical bytes, the same record traffic as the update's
        stale = U * (1.0 - U / N)
        return float(n * 4 + U * 4 + stale * 24 * logical)
    if name == "rlctr_ffm_fwd":
        return float(B * (F * 8 + F * 4 * logical + 4) + n * 4 * logical)
    return 0.0


def gemm_flops(key, m):
    """fp32-equivalent FLOPs of one dense-layer call (the 3xTF32 split issues 3x this on the tensor pipe)."""
    f = 2.0 * m["B"] * m["K"] * m["N"]
    if key.startswith("rlctr_linear_bwd"):
        return f * (2.0 if m.get("dx") else 1.0)
    return f


class Clocks:
    """nvidia-smi sampled DURING the timed region (B200_PROFILING.md 'clocks line')."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's CPU implementation, dense Adam, all host threads
# ----------------------------------------------------------------------------------------------
_REF = {"tried": False, "mod": None}


def reference_modules():
    """The reference's own ``src.models.p_model`` when its tree can be imported (never on the GPU box, which has no copy of it;
    in the build container it is /root/reference), else None -> the port in oracle/torch_port.py."""
    if _REF["tried"]:
        return _REF["mod"]
    _REF["tried"] = True
    for cand in (os.environ.get("RLCTR_REF_PATH"), "/root/reference", os.path.join(ROOT, "baseline", "_ref")):
        if cand and os.path.isfile(os.path.join(cand, "src", "models", "p_model.py")):
            try:
                sys.path.insert(0, cand)
                import importlib
                _REF["mod"] = importlib.import_module("src.models.p_model")
                break
            except Exception:
                sys.path.remove(cand)
    return _REF["mod"]


def cpu_kind():
    return "reference" if reference_modules() is not None else "port"


def cpu_models(N, D, names=MODELS):
    ref = reference_modules()
    torch.manual_seed(1)
    ms = []
    for name in names:
        if ref is not None:            # the reference's classes themselves (src/models/p_model.py)
            m = {"LR": lambda: ref.LR(N), "FM": lambda: ref.FM(N, D), "FFM": lambda: ref.FFM(N, F_FIELDS, D),
                 "DeepFM": lambda: ref.DeepFM(N, F_FIELDS, D)}[name]()
            opt = torch.optim.Adam(params=m.parameters(), lr=1e-3, weight_decay=1e-5)     # src/main/pretrain_main.py:181
        else:
            from oracle import torch_port as TP
            m = TP.PortCTR(name, N, F_FIELDS, D)
            opt = TP.make_adam(m)
        with torch.no_grad():
            for k, p in m.named_parameters():
                if "embedding" in k or k == "linear.weight":
                    p.mul_(0.1)
        m.train()
        ms.append((m, opt))
    return ms


def cpu_step(ms, x, y):
    lossf = torch.nn.BCELoss()
    yy = y.unsqueeze(1).float()
    for m, opt in ms:                   # the loop body of src/main/pretrain_main.py:96-102
        p = m(x)
        tl = lossf(p, yy)
        m.zero_grad()
        tl.backward()
        opt.step()
        tl.item()


def run_cpu(B, N, D, steps, warmup, names=MODELS, batch_fn=None):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    gen = torch.Generator().manual_seed(1)
    ms = cpu_models(N, D, names)
    batch_fn = batch_fn or make_batch
    batches = [batch_fn(gen, B, N, "cpu") for _ in range(min(steps + warmup, 4))]
    for i in range(warmup):
        cpu_step(ms, *batches[i % len(batches)])
    t0 = time.perf_counter()
    for i in range(steps):
        cpu_step(ms, *batches[(warmup + i) % len(batches)])
    dt = time.perf_counter() - t0
    return B * steps / dt, dt / steps, cores


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = max(int(args.gpus), 1)
    B, N, D = args.batch * world, args.rows, args.dims      # the B200 arm's GLOBAL batch (weak scaling: batch per GPU x N)
    # bound the run: one dense-Adam step costs O(N) on the CPU; time a probe step, then shrink N (which
    # only FAVOURS the reference: its step time is ~linear in N, SURVEY N3/H8) if K steps would not fit
    sample = f"full workload: global batch B={B}, N={N} rows, all three models, dense Adam"
    n_used = N
    probe_n = min(N, 1_000_000)
    _, t_probe, cores = run_cpu(B, probe_n, D, 1, 1)
    est = (t_probe * (0.3 + 0.7 * N / probe_n)) * (args.steps + args.warmup)
    if est > 200.0:
        n_used = max(int(N * 200.0 / est), 100_000)
        sample = (f"global batch B={B}, table rows reduced to N={n_used} (of {N}) so that {args.steps}+{args.warmup} steps end "
                  f"within minutes; the reference's step time grows with N, so this OVERSTATES its throughput")
    v, t_step, cores = run_cpu(B, n_used, D, args.steps, args.warmup)
    line = {"impl": "reference", "metric": "train samples/sec", "value": v, "unit": "samples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_step * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.batch, N, D, world),
            "cpu_baseline": {"value": v, "unit": "samples/s", "cores": cores, "kind": cpu_kind(), "sample": sample},
            "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def workload_config(B, N, D, world=1):
    return {"workload": "C2: LR+FM+DeepFM train step (fwd, BCE, bwd, Adam lr=1e-3 wd=1e-5, reference dense-Adam "
                        "numerics) on one batch" + ("" if world == 1 else f"; global batch split over {world} GPUs, tables row-sharded "
                        "(id mod G), dense parameters data-parallel"),
            "batch_per_gpu": B, "global_batch": B * world, "parallelism": "single GPU" if world == 1 else f"dp{world} x row-sharded tables",
            "fields": F_FIELDS, "latent_dims": D, "table_rows": N,
            "ids": "uniform over disjoint per-field ranges", "l2": "inputs larger than L2: 3 tables x 3 arrays x "
            f"{N * 4 * 12 / 1e6:.0f} MB touched at random rows, fresh batch every step"}


def table_layout(world, colocated):
    """How THIS implementation stores the tables (not part of the workload: the reference arm prints the same `config`)."""
    return ("co-located records: the three models' parameters + Adam moments of one id in one 384-byte record "
                       "(3 x 128-byte lines), one gather / catch-up / update per step for all three"
                       + ("" if world == 1 else "; the joint table row-sharded (id mod G), one per-sample exchange row of 128 bytes "
                          "all-gathered per step")
                       if colocated else "one fused-row table per model")


# ----------------------------------------------------------------------------------------------
# The other BASELINE.json configurations (SURVEY section 8d table) and the stock-PyTorch-on-B200 baseline
# ----------------------------------------------------------------------------------------------
CAMPAIGN_CARD = (24, 40, 300_000, 35, 370, 5, 25_000, 50_000, 21, 14, 4, 4, 130, 5)     # per-field cardinalities, rest -> usertag


def make_campaign_batch(gen, B, N, device):
    """C1 ids (SURVEY 8d): disjoint per-field ranges with campaign-like cardinalities, a Zipf-like (log-uniform rank: density
    ~ 1/rank) draw within a field, then a fixed random permutation of [0, N) (the first-seen rank interleaving of
    src/encode/data_.py); ~5 % positive labels.  Generated on the host (B is 4096) from a seed drawn off `gen`."""
    seed = int(torch.randint(0, 2 ** 31 - 1, (1,), generator=gen, device=gen.device).item())
    rng = np.random.default_rng(seed)
    card = list(CAMPAIGN_CARD)
    card.append(max(N - sum(card), 1))
    perm = np.random.default_rng(7).permutation(N)
    cols, base = [], 0
    for c in card:
        c = max(min(c, N - base), 1)
        rank = np.minimum(np.floor(np.power(float(c), rng.random(B))).astype(np.int64) - 1, c - 1)
        cols.append(base + np.maximum(rank, 0))
        base += c
    x = perm[np.minimum(np.stack(cols, axis=1), N - 1)]
    y = (rng.random(B) < 0.05).astype(np.int64)
    return torch.as_tensor(x).to(device), torch.as_tensor(y).to(device)


def _time_steps(ctx, run, steps, warmup, after=None):
    """(ms per step, max over ranks): CUDA events around `steps` calls of run(i) after `warmup` untimed ones; `after()`
    (e.g. the lazy flush) runs inside the timed region."""
    for i in range(warmup):
        run(i)
    ctx["barrier"]()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        run(warmup + i)
    if after is not None:
        after()
    e1.record()
    ctx["barrier"]()
    return ctx["max_over_ranks"](e0.elapsed_time(e1)) / steps


def _hbm(bytes_per_sample, samples_per_s, peak, what):
    a = bytes_per_sample * samples_per_s / 1e9
    return {"bound": "hbm", "algorithmic_bytes_per_sample": bytes_per_sample, "achieved": a, "peak": peak, "unit": "GB/s",
            "frac": a / peak, "what": what}


def run_c1(ctx):
    """configs[0]: the reference's own CPU-runnable case -- FM, B=4096, N=1e6, campaign-shaped ids -- on the B200 path and,
    beside it, the reference's CPU implementation on the host cores."""
    from rl_ctr_prediction_b200 import graphs, optim, p_model
    dev = ctx["dev"]
    B, N, D = 4096, 1_000_000, 10
    gen = torch.Generator(device=dev).manual_seed(11)
    m = p_model.FM(N, D, device=dev)
    with torch.no_grad():
        m.table.mul_(0.1)
    m.train()
    opt = optim.Adam(m.parameters(), lr=1e-3, weight_decay=1e-5)
    step = graphs.GraphedTrainStep([(m, opt)], torch.nn.BCELoss())
    batches = [make_campaign_batch(gen, B, N, dev) for _ in range(16)]
    steps = 200
    ms = _time_steps(ctx, lambda i: step(*batches[i % len(batches)]), steps, 8, after=m.flush)
    v = B / (ms / 1e3)
    out = {"workload": "C1: FM train step, B=4096, F=15, D=10, N=1e6, campaign-shaped Zipf ids (SURVEY 8d), graph replay, lazy "
                       "flush inside the timed region", "value": v, "unit": "samples/s", "ms_per_step": ms, "steps": steps,
           "roofline": _hbm(6068, v, ctx["peak"], "FM train step, sparse/lazy update (SURVEY 8d): at B=4096 the step is "
                                                  "launch-latency bound (a handful of ~5 us kernels), not HBM bound")}
    del m, opt, step
    try:
        vc, t_step, cores = run_cpu(B, N, D, 10, 3, names=("FM",), batch_fn=make_campaign_batch)
        out["cpu_reference"] = {"value": vc, "unit": "samples/s", "cores": cores, "kind": cpu_kind(), "ms_per_step": t_step * 1e3,
                                "sample": "10 steps after 3 warm-up, dense Adam over all 1e6 rows (reference semantics)"}
    except Exception as exc:
        out["cpu_reference"] = {"error": str(exc)[:200]}
    return out


def _frozen_ctr_models(N, D, dev, names=("LR", "FM", "FFM")):
    from rl_ctr_prediction_b200 import p_model
    md = {}
    for i, name in enumerate(names):
        m = {"LR": lambda: p_model.LR(N, device=dev), "FM": lambda: p_model.FM(N, D, device=dev),
             "FFM": lambda: p_model.FFM(N, F_FIELDS, D, device=dev)}[name]()
        with torch.no_grad():
            m.table.mul_(0.1)
        md[i] = m.eval()
    return md


def _policy_flops(widths):
    return 2.0 * sum(a * b for a, b in zip(widths[:-1], widths[1:]))


def run_c3(ctx):
    """configs[2]: REINFORCE policy over model_dict = {LR, FM, FFM} (src/all_main/main.py:437), reward from generate_preds,
    the update fused into the step (PG_model.PolicyGradient.fused_step), one CUDA graph."""
    from rl_ctr_prediction_b200 import PG_model, graphs
    dev, args = ctx["dev"], ctx["args"]
    B, N, D = args.batch, args.rows, args.dims
    md = _frozen_ctr_models(N, D, dev)
    M = len(md)
    torch.manual_seed(3)
    pg = PG_model.PolicyGradient(N, F_FIELDS, D, action_nums=M - 1, device=dev)
    with torch.no_grad():
        pg.policy_net.embedding_layer.table.mul_(0.1)
    gen = torch.Generator(device=dev).manual_seed(13)
    batches = [make_batch(gen, B, N, dev) for _ in range(8)]
    step = graphs.GraphedCallable(lambda x, y: pg.fused_step(x, y.reshape(-1, 1), md)[0], [pg.optimizer])
    steps = 20
    ms = _time_steps(ctx, lambda i: step(*batches[i % len(batches)]), steps, 5)
    v = B / (ms / 1e3)
    P = F_FIELDS * (F_FIELDS - 1) // 2
    hbm_bytes = 1740 + 184 + 784 + 8584 + (12 * M + 24)       # state encoder + LR, FM, FFM forwards + generate_preds (SURVEY 8d)
    fl = 3.0 * _policy_flops([P + F_FIELDS * D, 1024, 512, 256, 128, M - 1])          # forward + dgrad + wgrad
    tf = fl * v / 1e12
    return {"workload": "C3: Feature_Embedding -> policy MLP (255-1024-512-256-128-2, ReLU, Dropout .2) -> action draw -> "
                        "generate_preds over {LR, FM, FFM} (N=1e7 rows each) -> +-1 reward -> returns -> REINFORCE loss -> Adam "
                        "(lr 1e-4, wd 1e-5), B=65536, one CUDA graph, nothing leaves the device",
            "value": v, "unit": "samples/s", "ms_per_step": ms, "steps": steps, "graph_launches_per_step": step.launches_per_step,
            "roofline": {"bound": "tensor", "fp32_equiv_flop_per_sample": fl, "achieved": tf, "peak": ctx["tpeak"], "unit": "TFLOP/s",
                         "frac": tf / ctx["tpeak"], "tensor_pipe_issued_TFLOPs": 3 * tf, "tensor_pipe_issued_frac": 3 * tf / ctx["tpeak"],
                         "what": "policy MLP GEMMs (3xTF32: 3 tensor-pipe MMAs per fp32 product), 5.7 MFLOP/sample against "
                                 "11.4 KB/sample of HBM gathers: the step is tensor-bound",
                         "hbm": _hbm(hbm_bytes, v, ctx["peak"], "state encoder + LR/FM/FFM scoring gathers + generate_preds")}}


def run_c4(ctx):
    """configs[3]: FFM + DeepFM, N=1e7-row tables; one GPU: fused-row tables in HBM; N>1: row-sharded over the GPUs."""
    from rl_ctr_prediction_b200 import graphs, optim, p_model
    dev, args, world = ctx["dev"], ctx["args"], ctx["world"]
    B, N, D = args.batch, args.rows, args.dims
    ms_ = []
    for name in ("FFM", "DeepFM"):
        if world > 1:
            from rl_ctr_prediction_b200 import sharded
            m = sharded.ShardedCTR(name, N, F_FIELDS, D, device=dev)
        else:
            m = p_model.FFM(N, F_FIELDS, D, device=dev) if name == "FFM" else p_model.DeepFM(N, F_FIELDS, D, device=dev)
        with torch.no_grad():
            m.table.mul_(0.1)
        m.train()
        ms_.append((m, optim.Adam(m.parameters(), lr=1e-3, weight_decay=1e-5, mode="lazy")))
    gen = torch.Generator(device=dev).manual_seed(17 + ctx["rank"])
    batches = [make_batch(gen, B, N, dev) for _ in range(8)]
    step = graphs.GraphedTrainStep(ms_, torch.nn.BCELoss(), fork=False)
    steps = 20

    def flush():
        for m, _ in ms_:
            m.flush()
    ms = _time_steps(ctx, lambda i: step(*batches[i % len(batches)]), steps, 5, after=flush)
    v = B * world / (ms / 1e3)
    return {"workload": f"C4: FFM + DeepFM train step, B={B} per GPU, F=15, D=10, N=1e7 rows per table (FFM row = 151 floats), "
                        + ("single GPU" if world == 1 else f"tables row-sharded over {world} GPUs (id mod G)")
                        + ", graph replay, lazy flush inside the timed region",
            "value": v, "unit": "samples/s", "ms_per_step": ms, "steps": steps, "n_gpus": world,
            "roofline": _hbm(76268 + 6068, v / world, ctx["peak"], "FFM train 76,268 B/sample + FM-part of DeepFM 6,068 B/sample "
                                                                   "(SURVEY 8d), per GPU; DeepFM's tower is tensor work on top")}


def run_c5(ctx):
    """configs[4]: the full src/all_main/main.py step (state encoder, DDQN + DDPG acting, generate_preds over {LR, FM, FFM},
    replay store, DDQN learn, DDPG critic + actor learn, Polyak) at a global batch of 1M; N>1: strong scaling, the batch
    split over the ranks, frozen tables replicated, policy nets data-parallel (all-reduced gradients, cross-rank BatchNorm)."""
    from rl_ctr_prediction_b200 import all_main
    from rl_ctr_prediction_b200.DDQN_model import RingMemory
    from rl_ctr_prediction_b200.Feature_embedding import Feature_Embedding
    dev, args, world = ctx["dev"], ctx["args"], ctx["world"]
    N, D = args.rows, args.dims
    B_global = 1 << 20
    B = B_global // world
    md = _frozen_ctr_models(N, D, dev)
    M = len(md)
    torch.manual_seed(5)
    fe = Feature_Embedding(N, F_FIELDS, D, device=dev)
    with torch.no_grad():
        fe.table.mul_(0.1)
    ddqn, ddpg = all_main.get_model(M, N, F_FIELDS, D, 256, 1 << 21, dev, "1458")
    if world > 1:
        if os.environ.get("RLCTR_RL_DP", "gather") == "gather":
            all_main.make_gathered_replay(ddqn, ddpg)         # one all_gather of the replay draws per agent, replicated learn step
        else:
            all_main.make_data_parallel(ddqn, ddpg)           # cross-rank BatchNorm + averaged gradients (a collective per layer)
    RingMemory.device_sampling = True                     # replay indices drawn on the device (SURVEY 8f.4): no host RNG round trip
    ddqn.device_rng = ddpg.device_rng = True              # exploration draws on the device too (the reference: CPU rand + H2D)
    gen = torch.Generator(device=dev).manual_seed(19 + ctx["rank"])
    batches = [make_batch(gen, B, N, dev) for _ in range(3)]
    steps = 5

    def run(i):
        x, y = batches[i % len(batches)]
        all_main.train_step(ddqn, ddpg, md, x, y.reshape(-1, 1), fe, 0.9, dev)
    try:
        ms = _time_steps(ctx, run, steps, 2)
    finally:
        RingMemory.device_sampling = False
    v = B_global / (ms / 1e3)
    P = F_FIELDS * (F_FIELDS - 1) // 2
    S = P + F_FIELDS * D
    fl = _policy_flops([S, 300, 300, 300, M - 1]) + _policy_flops([S + 1, 300, 300, 300, M])     # acting: DDQN + Actor forwards
    tf = fl * v / 1e12
    hbm_bytes = 1740 + 184 + 784 + 8584 + (12 * M + 24) + 4 * (F_FIELDS + 2) + 4 * (F_FIELDS + M + 2)
    return {"workload": f"C5: src/all_main step, global batch {B_global} ({B} per GPU), N=1e7-row frozen tables, M=3 CTR models, "
                        "replay batch 256, eager launches (the step reads td_error / a_loss on the host like the reference)"
                        + ("" if world == 1 else "; acting data-parallel over the batch, frozen tables replicated, the ranks' replay "
                           "draws joined by one all_gather per agent and the learn step replicated (== the single-process step on the "
                           "joined batch, BatchNorm statistics included; all_main.make_data_parallel is the gradient-all-reduce form)"),
            "value": v, "unit": "samples/s", "ms_per_step": ms, "steps": steps, "n_gpus": world, "scaling": "strong",
            "roofline": {"bound": "tensor", "fp32_equiv_flop_per_sample": fl, "achieved": tf, "peak": ctx["tpeak"] * world,
                         "unit": "TFLOP/s", "frac": tf / (ctx["tpeak"] * world), "tensor_pipe_issued_TFLOPs": 3 * tf,
                         "tensor_pipe_issued_frac": 3 * tf / (ctx["tpeak"] * world),
                         "what": "acting-path GEMMs of the DDQN and the DDPG actor over the whole batch (eval-mode BatchNorm folded "
                                 "into the layers); the learn steps run on 256-sample replay batches",
                         "hbm": _hbm(hbm_bytes, v / world, ctx["peak"], "state encoder + three scoring gathers + generate_preds + "
                                                                        "replay stores, per GPU")}}


def run_eager_gpu(dev, B, N, D, our_value):
    """BASELINE.md section 1 names it first: the stock-PyTorch path on the same box.  The reference's modules restated on stock
    ATen ops (oracle/torch_port.PortCTR == src/models/p_model.py) moved to the B200, the reference's loop body, dense
    torch.optim.Adam over all rows -- what `python src/main/pretrain_main.py --device cuda:0` does per batch."""
    from oracle import torch_port as TP
    torch.manual_seed(1)
    ms = []
    for name in MODELS:
        m = TP.PortCTR(name, N, F_FIELDS, D).to(dev)
        with torch.no_grad():
            for k, p in m.named_parameters():
                if "embedding" in k or k == "linear.weight":
                    p.mul_(0.1)
        m.train()
        ms.append((m, torch.optim.Adam(m.parameters(), lr=1e-3, weight_decay=1e-5)))
    gen = torch.Generator(device=dev).manual_seed(1)
    batches = [make_batch(gen, B, N, dev) for _ in range(4)]
    lossf = torch.nn.BCELoss()

    def step(i):
        x, y = batches[i % len(batches)]
        yy = y.unsqueeze(1).float()
        for m, opt in ms:
            tl = lossf(m(x), yy)
            m.zero_grad()
            tl.backward()
            opt.step()
    for i in range(3):
        step(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    steps = 8
    e0.record()
    for i in range(steps):
        step(3 + i)
    e1.record()
    torch.cuda.synchronize()
    ms_step = e0.elapsed_time(e1) / steps
    v = B / (ms_step / 1e3)
    return {"value": v, "unit": "samples/s", "ms_per_step": ms_step, "steps": steps, "speedup_of_this_repo": our_value / v,
            "impl": "stock PyTorch eager on cuda:0: nn.Embedding gathers, autograd (dense embedding gradients), "
                    "torch.optim.Adam(lr=1e-3, weight_decay=1e-5) over all rows; same workload (C2), fp32, TF32 off"}


DUMP_ROWS = 1 << 16        # table rows sampled by --dump-outputs
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, ms, losses, n_rows):
    """--dump-outputs: the last timed step's loss of every model and, after the flush, its parameters under the reference's
    state_dict keys, as float32 (integers as float64) .npy files.  Dense tensors are written whole; of the tables (n_rows
    rows) the same fixed, seeded sample of rows, listed in table_rows.npy.  Two builds run with the same arguments can
    then be compared file by file."""
    os.makedirs(out_dir, exist_ok=True)
    rows = np.random.default_rng(0).choice(n_rows, size=min(n_rows, DUMP_ROWS), replace=False)
    rows.sort()
    out = {"table_rows": rows.astype(np.float64)}
    models = []
    for m, _ in ms:                       # a co-located group holds LR, FM, DeepFM as its members, in that order
        models.extend(m.members if hasattr(m, "members") else [m])
    loss = torch.cat([l.reshape(-1) for l in losses]).cpu().numpy()
    assert len(models) == loss.size == len(MODELS), (len(models), loss.size)
    idx = None
    for name, m, l in zip(MODELS, models, loss):
        out[f"{name}.loss"] = np.float32(l)
        for key, t in m.state_dict().items():
            if t.dim() > 0 and t.shape[0] == n_rows:
                if idx is None:
                    idx = torch.as_tensor(rows, device=t.device)
                t = t[idx]
            a = t.cpu().numpy()
            out[f"{name}.{key}"] = a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)
    total = sum(a.nbytes for a in out.values())
    assert total <= DUMP_MAX_BYTES, f"--dump-outputs would write {total} bytes"
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    torch.cuda.empty_cache()


# ----------------------------------------------------------------------------------------------
# B200 arm
# ----------------------------------------------------------------------------------------------
def b200_arm(args):
    import torch.distributed as dist
    from rl_ctr_prediction_b200 import _lib, optim, p_model, pretrain_main as PM

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if args.dump_outputs:
            raise SystemExit("--dump-outputs runs on one GPU")
        dist.init_process_group("nccl", device_id=dev)
    B, N, D, K, W = args.batch, args.rows, args.dims, args.steps, args.warmup
    W = max(W, 3)
    lib = _lib.load()
    torch.manual_seed(1 + rank)
    gen = torch.Generator(device=dev).manual_seed(1 + rank)

    colocate = not args.no_colocate

    def build_models(colocated=None):
        if (colocate if colocated is None else colocated) and world > 1:
            # the co-located record row-sharded over the GPUs (sharded.ShardedGroup): one routed view, one remote gather, one
            # all_gather of per-sample rows, one push, one all_reduce, one update per step for the three models
            from rl_ctr_prediction_b200 import sharded
            group = sharded.ShardedGroup(MODELS, N, F_FIELDS, D, device=dev)
            with torch.no_grad():
                group.table.mul_(0.1)
            group.train()
            return [(group, optim.Adam(group.parameters(), lr=1e-3, weight_decay=1e-5, mode="lazy"))]
        if colocate if colocated is None else colocated:
            # one record per id for the three models (colocated.py): one gather, one catch-up, one update per step
            from rl_ctr_prediction_b200 import colocated as _co
            members = [p_model.LR(N, device=dev), p_model.FM(N, D, device=dev), p_model.DeepFM(N, F_FIELDS, D, device=dev)]
            with torch.no_grad():
                for m in members:
                    m.table.mul_(0.1)
                    m.train()
            group = _co.colocate(members)
            del members
            torch.cuda.empty_cache()
            group.train()
            return [(group, optim.Adam(group.parameters(), lr=1e-3, weight_decay=1e-5, mode="lazy"))]
        ms = []
        for name in MODELS:
            if world > 1:      # BASELINE.json configs[3]: tables row-sharded over the GPUs (peer-mapped shards over NVLink)
                from rl_ctr_prediction_b200 import sharded
                own = not args.no_fork                      # a communicator per model: the models can be graph branches
                m = sharded.ShardedCTR(name, N, F_FIELDS, D, device=dev,
                                       group=dist.new_group(list(range(world))) if own else None)
                m.fork_ok = own
            else:
                m = {"LR": lambda: p_model.LR(N, device=dev), "FM": lambda: p_model.FM(N, D, device=dev),
                     "DeepFM": lambda: p_model.DeepFM(N, F_FIELDS, D, device=dev)}[name]()
            with torch.no_grad():
                m.table.mul_(0.1)
            m.train()
            ms.append((m, optim.Adam(m.parameters(), lr=1e-3, weight_decay=1e-5, mode="lazy")))
        return ms

    lossf = torch.nn.BCELoss()

    def step(ms, x, y):
        # the eager form of exactly what the CUDA graph replays (graphs.eager_step): the fused loss head for every model, autograd
        # for DeepFM's tower, the sharded step for N > 1
        from rl_ctr_prediction_b200 import graphs as _g
        return [_g.eager_step(m, opt, lossf, x, y) for m, opt in ms]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident timing (`value`) -------------------------------------
    # The whole three-model step is one CUDA graph (rl_ctr_prediction_b200/graphs.py): two eager warm-up steps, capture
    # at the third, replays after that.  N > 1: the sharded step has no host synchronisation either (fixed-size id
    # all_gather, device barriers), so it is captured the same way.
    ms = build_models()
    batches = [make_batch(gen, B, N, dev) for _ in range(K + W)]
    use_graph = not args.no_graph
    if use_graph:
        from rl_ctr_prediction_b200 import graphs
        gstep = graphs.GraphedTrainStep(ms, lossf, fork=not args.no_fork)
        run_step = lambda x, y: gstep(x, y)
    else:
        gstep = None
        run_step = lambda x, y: step(ms, x, y)
    clocks = Clocks(local)
    clocks.start()                       # sampled from the warm-up on: the timed region itself lasts tens of milliseconds
    for i in range(W):
        run_step(*batches[i])
    barrier()
    l0 = lib.rlctr_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        losses = run_step(*batches[W + i])
    for m, _ in ms:
        m.flush()
    e1.record()
    barrier()
    launches = lib.rlctr_launch_count() - l0
    if gstep is not None and gstep.graph is not None:
        launches += gstep.launches_per_step * K          # replayed launches are not seen by the host-side tally
    clk = clocks.stop()
    ms_total = e0.elapsed_time(e1)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ms, losses, N)

    def max_over_ranks(v):
        t = torch.tensor([v], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    ms_total = max_over_ranks(ms_total)
    value = B * K * world / (ms_total / 1e3)

    # ---------------- steady state: windows of 20 steps WITHOUT the flush, then the flush on its own -----------------
    # (the headline above charges one full flush of all three tables to K steps; an epoch of the reference is ~500 steps
    # per flush, so the per-step cost of the lazy mode in production is the window figure plus flush_ms / steps_per_epoch)
    steady = None
    if args.windows > 0:
        win, per_window = 20, []
        for w in range(args.windows):
            barrier()
            e0.record()
            for i in range(win):
                run_step(*batches[(w * win + i) % len(batches)])
            e1.record()
            barrier()
            per_window.append(max_over_ranks(e0.elapsed_time(e1)) / win)
        barrier()
        e0.record()
        for m, _ in ms:
            m.flush()
        e1.record()
        barrier()
        flush_ms = max_over_ranks(e0.elapsed_time(e1))
        med = statistics.median(per_window)
        steady = {"value": B * world / (med / 1e3), "unit": "samples/s", "ms_per_step": med, "windows": args.windows,
                  "steps_per_window": win, "ms_per_step_by_window": [round(v, 4) for v in per_window], "flush_ms": flush_ms,
                  "note": "graph replay, no flush inside the windows (row staleness has reached its stationary level after the "
                          "first ~30 steps); flush_ms = settling all rows of all three tables once (end of epoch / state_dict)"}

    # ---------------- per-kernel pass: the same steps, eagerly, CUDA events around every library call --------------
    prof = _lib.KernelTimer()
    Kp = min(K, args.profile_steps)
    _lib.set_timer(prof)
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for i in range(Kp):
        step(ms, *batches[W + i])
    for m, _ in ms:
        m.flush()
    p1.record()
    barrier()
    _lib.set_timer(None)
    ms_prof = p0.elapsed_time(p1)

    # ---------------- roofline of the dominant kernel --------------------------------------
    kern = prof.summary(alg_bytes)   # name -> (launches, mean ms, algorithmic bytes per launch)
    peak, peak_src = peaks()
    tpeak, tpeak_src = tensor_peak()
    gemm = {}
    groups = {}                      # library entry point (all models) -> total ms in the profiled pass
    for k, (n_l, mean_ms, alg) in kern.items():
        groups[k.split("[")[0]] = groups.get(k.split("[")[0], 0.0) + n_l * mean_ms
    for k in list(kern):
        if k.startswith("rlctr_linear"):
            n_l, mean_ms, _ = kern.pop(k)
            fl = sum(gemm_flops(k, m) for _, _, m in prof.records[k]) / n_l
            gemm[k] = {"launches": n_l, "mean_ms": mean_ms, "fp32_equiv_TFLOPs": fl / (mean_ms / 1e3) / 1e12,
                       "tensor_pipe_TFLOPs_3x": 3 * fl / (mean_ms / 1e3) / 1e12}
    all_kernels = {k: {"launches": v[0], "mean_ms": v[1], "GBps": v[2] / (v[1] / 1e3) / 1e9 if v[1] > 0 else None,
                       "frac_of_hbm_peak": v[2] / (v[1] / 1e3) / 1e9 / peak if v[1] > 0 else None,
                       "ncu_dram_bytes_per_launch": NCU_TRAFFIC.get(k)}
                   for k, v in kern.items()}
    step_ms = ms_total / K                                # the graph-replay step the shares are read against
    shares = {g: round(tms / Kp / step_ms, 4) for g, tms in sorted(groups.items(), key=lambda kv: -kv[1])}
    top = max(groups, key=groups.get) if groups else None
    roof = None
    if top is not None and top.startswith("rlctr_linear"):
        keys = [k for k in gemm if k.startswith(top)]
        tot_ms = sum(gemm[k]["launches"] * gemm[k]["mean_ms"] for k in keys)
        tot_fl = sum(gemm_flops(k, m) for k in keys for _, _, m in prof.records[k])
        achieved = tot_fl / (tot_ms / 1e3) / 1e12           # ALGORITHMIC (fp32-equivalent) FLOP/s: 2*B*K*N per GEMM (SURVEY 8d)
        roof = {"bound": "tensor", "kernel": top + " (gemm3x_tma_kernel: all tower layers)", "achieved": achieved, "peak": tpeak,
                "unit": "TFLOP/s", "frac": achieved / tpeak, "tensor_pipe_issued_TFLOPs": 3 * achieved,
                "tensor_pipe_issued_frac": 3 * achieved / tpeak, "traffic": NCU_TRAFFIC.get(top),
                "traffic_note": "DRAM bytes (ncu dram__bytes_read+write) of ALL kernels of this entry point in one step, B=65536 "
                                "(profiles/r2f_ncu_top_kernels.md; re-captured on the final build, same figures within 1 %: profiles/r2r_ncu_gemm.md); "
                                "achieved / peak are FLOP rates over the same kernels",
                "peak_source": tpeak_src,
                "flops_counted": "algorithmic fp32-equivalent FLOPs; the 3xTF32 split issues 3 tf32 MMAs per product "
                                 "(tensor_pipe_issued_*)", "share_of_step": groups[top] / Kp / step_ms}
    elif top is not None:
        keys = [k for k in kern if k.split("[")[0] == top]
        key = max(keys, key=lambda k: kern[k][0] * kern[k][1])        # the heaviest launch of the dominant entry point
        n_l, mean_ms, alg = kern[key]
        achieved = alg / (mean_ms / 1e3) / 1e9
        roof = {"bound": "hbm", "kernel": key, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": NCU_TRAFFIC.get(key), "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg, "launches_timed": n_l, "mean_ms": mean_ms,
                "share_of_step": groups[top] / Kp / step_ms}
    if roof is not None and world > 1:
        # NVLink side of the sharded step (north_star: throughput as a fraction of the HBM / NVLink roofline): ALGORITHMIC bytes a
        # rank receives per step -- logical row sizes, as for HBM -- against the measured 770 GB/s per direction peer rate
        n_occ, rho = B * F_FIELDS, (world - 1) / world
        logical = {"LR": 1, "FM": D + 1, "DeepFM": D + 1}
        fwd = {m: rho * n_occ * 4 * logical[m] for m in MODELS}                     # remote rows read by the forward gathers
        rows_rs = 16 if D <= 15 else (D + 1 + 3) // 4 * 4
        gath = {"LR": (world - 1) * B * 4, "FM": (world - 1) * B * 4 * rows_rs, "DeepFM": (world - 1) * B * 4 * rows_rs}
        push = rho * n_occ * D * 4                                                   # DeepFM's tower-input gradients, pushed to the owners
        route = rho * n_occ * 8                                                      # (local row, global slot) pairs written to the owners
        if colocate:                                                                 # one joint gather, one exchange row per sample
            fwd = {"group": rho * n_occ * 4 * sum(logical.values())}
            gath = {"group": (world - 1) * B * 4 * 32}
        total = sum(fwd.values()) + sum(gath.values()) + push + route
        nv_peak = 770.0
        per_kernel = {}
        for m in (["group"] if colocate else MODELS):
            k = "rlctr_group_fwd[ShardedGroup]" if colocate else f"rlctr_embed_fwd[Sharded{m}]"
            if k in kern and kern[k][1] > 0:
                gbps = fwd[m] / (kern[k][1] / 1e3) / 1e9
                per_kernel[k] = {"nvlink_bytes": fwd[m], "mean_ms": kern[k][1], "GBps": gbps, "frac": gbps / nv_peak}
        if "rlctr_push_rows" in kern and kern["rlctr_push_rows"][1] > 0:
            gbps = push / (kern["rlctr_push_rows"][1] / 1e3) / 1e9
            per_kernel["rlctr_push_rows"] = {"nvlink_bytes": push, "mean_ms": kern["rlctr_push_rows"][1], "GBps": gbps, "frac": gbps / nv_peak}
        if "rlctr_route_ids" in kern and kern["rlctr_route_ids"][1] > 0:
            gbps = route / (kern["rlctr_route_ids"][1] / 1e3) / 1e9
            per_kernel["rlctr_route_ids"] = {"nvlink_bytes": route, "mean_ms": kern["rlctr_route_ids"][1], "GBps": gbps, "frac": gbps / nv_peak}
        step_gbps = total / (step_ms / 1e3) / 1e9
        roof["nvlink"] = {"bytes_received_per_step_per_gpu": total, "achieved": step_gbps, "peak": nv_peak, "unit": "GB/s",
                          "frac": step_gbps / nv_peak, "nvlink_frac": step_gbps / nv_peak,
                          "peak_source": "measured peer copy, 770 GB/s per direction per GPU (B200_PROFILING.md); 900 nominal",
                          "breakdown_bytes": {"forward_remote_rows": sum(fwd.values()), "all_gather_sums_dlogit": sum(gath.values()),
                                              "push_tower_input_grads": push, "route_ids": route},
                          "kernels": per_kernel,
                          "note": "whole-step figure: the step is not NVLink-bound (the exchanges overlap HBM- and tensor-bound "
                                  "work on other graph branches); `kernels` are the NVLink-bound launches on their own"}
    if roof is not None:
        roof["share_of_step_by_entry_point"] = shares
        roof["profiled_pass"] = {"steps": Kp, "ms_per_step": ms_prof / Kp, "mode": "eager, CUDA events around every library call"}
        roof["all_kernels"] = all_kernels
    del ms, batches
    torch.cuda.empty_cache()

    # ---------------- end to end through the drop-in API (`e2e`) ---------------------------
    e2e = None
    if not args.no_e2e:
        ms = build_models()
        gen_c = torch.Generator().manual_seed(100 + rank)
        host = []
        for _ in range(K + W):
            x, y = make_batch(gen_c, B, N, "cpu")
            host.append((x.pin_memory(), y.pin_memory()))

        def e2e_step_eager(xh, yh):
            x = xh.to(dev, non_blocking=True)
            y = torch.unsqueeze(yh, 1).to(dev, non_blocking=True)
            total = 0.0
            for m, opt in ms:
                if world > 1:
                    total += m.train_step(x, yh.to(dev, non_blocking=True), opt).sum().item()
                    continue
                p = m(x)                                   # src/main/pretrain_main.py:96-103, per model
                tl = lossf(p, y.float())
                m.zero_grad()
                tl.backward()
                opt.step()
                total += tl.item()                         # device -> host read of the step's loss
            return total

        def timed(run):
            barrier()
            e0.record()
            run()
            for m, _ in ms:
                m.flush()
            e1.record()
            barrier()
            t = torch.tensor([max(e0.elapsed_time(e1), 0.0)], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return t.item()

        bytes_in, bytes_out = B * F_FIELDS * 8 + B * 8, 4 * len(MODELS)
        if use_graph:
            # the public call: GraphedTrainStep on pinned HOST batches; the copy of batch i+1 is issued before step i
            # (graphs.GraphedTrainStep.prefetch) and every step's three losses are read back to the host
            from rl_ctr_prediction_b200 import graphs
            gs = graphs.GraphedTrainStep(ms, lossf, fork=not args.no_fork)
            sink = []

            def run_graphed(lo, hi):
                h = gs.prefetch(*host[lo])
                pending = None
                for i in range(lo, hi):
                    nxt = gs.prefetch(*host[i + 1]) if i + 1 < hi else None
                    fetch = gs.losses_to_host(gs(h))               # device -> host copy of this step's three losses
                    if pending is not None:
                        sink.append(pending())                     # read step i-1 on the host while step i runs
                    pending, h = fetch, nxt
                sink.append(pending())

            run_graphed(0, W)
            ms_e2e = timed(lambda: run_graphed(W, W + K))
            e2e = {"value": B * K * world / (ms_e2e / 1e3), "unit": "samples/s", "h2d_bytes_per_step": bytes_in,
                   "d2h_bytes_per_step": bytes_out, "ms_per_step": ms_e2e / K,
                   "api": "graphs.GraphedTrainStep: step.prefetch(pinned host features, labels); losses = step(handle); "
                          "every step's losses copied to pinned host memory and read there one step later"}
            del gs
            ms = None
            torch.cuda.empty_cache()
            ms = build_models(colocated=False if world == 1 else None)   # one GPU: the reference's per-model loop body
        elif colocate and world == 1:
            ms = None
            torch.cuda.empty_cache()
            ms = build_models(colocated=False)
        for i in range(W):
            e2e_step_eager(*host[i])
        ms_eager = timed(lambda: [e2e_step_eager(*host[W + i]) for i in range(K)])
        eager = {"value": B * K * world / (ms_eager / 1e3), "unit": "samples/s", "h2d_bytes_per_step": bytes_in,
                 "d2h_bytes_per_step": bytes_out, "ms_per_step": ms_eager / K,
                 "api": "model(x); nn.BCELoss; zero_grad; backward; optim.Adam.step; loss.item()  (the reference's loop body, "
                        "launched eagerly from Python: host-bound)"}
        if e2e is None:
            e2e = eager
        else:
            e2e["dropin_eager_loop"] = eager
        del ms, host
        torch.cuda.empty_cache()

    # ---------------- CPU baseline (rank 0, N=1 only) ---------------------------------------
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        v, t_step, cores = run_cpu(B, N, D, args.cpu_steps, 1)
        cpu = {"value": v, "unit": "samples/s", "cores": cores, "kind": cpu_kind(),
               "sample": f"{args.cpu_steps} steps (after 1 warm-up) of the same workload (B={B}, N={N}), "
                         f"{t_step:.2f} s/step, dense Adam over all rows (reference semantics)"}

    # ---------------- the other BASELINE.json configurations + the stock-PyTorch-on-B200 baseline ------------------
    configs, eager_gpu = None, None
    if not args.no_configs:
        configs = {}
        ctx = {"dev": dev, "world": world, "rank": rank, "barrier": barrier, "max_over_ranks": max_over_ranks, "peak": peaks()[0],
               "tpeak": tensor_peak()[0], "args": args}
        for name in [c.strip() for c in args.configs.split(",") if c.strip()]:
            fn = {"C1": run_c1, "C3": run_c3, "C4": run_c4, "C5": run_c5}.get(name)
            if fn is None or (world > 1 and name in ("C1", "C3")):
                continue                                  # C1 / C3 are single-GPU configurations
            try:
                configs[name] = fn(ctx)
            except Exception as exc:                      # a config that cannot run must not take the headline down with it
                configs[name] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
            torch.cuda.empty_cache()
    if world == 1 and not args.no_eager_gpu:
        try:
            eager_gpu = run_eager_gpu(dev, B, N, D, value)
        except Exception as exc:
            eager_gpu = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        torch.cuda.empty_cache()

    if rank == 0:
        line = {"metric": "train samples/sec", "value": value, "unit": "samples/s", "n_gpus": world, "steps": K,
                "warmup": W, "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(B, N, D, world), "table_layout": table_layout(world, colocate),
                "roofline": roof, "gemm": gemm, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clk,
                "cuda_graph": bool(use_graph), "graph_branches": bool(use_graph and not args.no_fork),
                "steady_state": steady, "configs": configs, "gpu_eager_baseline": eager_gpu}
        print(json.dumps(line))
    if world > 1:
        torch.cuda.synchronize()
        sys.stdout.flush()
        os._exit(0)           # symmetric-memory mappings are released with the process; no collective teardown


def main():
    args = parse()
    if args.impl == "reference":
        reference_arm(args)
    else:
        b200_arm(args)


if __name__ == "__main__":
    main()
