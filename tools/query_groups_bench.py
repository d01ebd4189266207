#!/usr/bin/env python
"""Query groups vs link pairs on the citation2 eval workload: one JSON line.

The citation2 eval sends, per query, one source and K = 1 + negs candidate targets.  LinkScoreStream.score takes them
as int64 pairs [2, L] (16 bytes per link); score_grouped takes source [Q] and targets [Q, K] (4 or 8 bytes per link
plus one id per query) and expands each batch on the device.  This script times, in one process and on bench.py's
seeded workload and default batch (2,048 queries x 1,001 links per step), alternating the forms call by call:

  dev_pairs, dev_grouped_i32                   inputs resident on the device (the device step)
  e2e_pairs, e2e_grouped_i64, e2e_grouped_i32  inputs in pinned host memory, scores to pinned host memory (out_host)

Per form: ms_per_step (total time over every timed batch), its spread over the timed calls (min / median / max
ms_per_step of one call of --steps batches), links_per_s (all ranks) and h2d_bytes_per_step (ids shipped to the device,
from the shapes).  Also: max |score difference| of every form against dev_pairs, world size, and the GPU's name,
power limit and max SM clock (read-only nvidia-smi query in the same run).

  python tools/query_groups_bench.py [--steps 20 --warmup 3 --batches 200]
  torchrun --nproc_per_node N tools/query_groups_bench.py     (every rank scores its own queries, as bench.py)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

import bench as B  # noqa: E402

FORMS = ("dev_pairs", "dev_grouped_i32", "e2e_pairs", "e2e_grouped_i64", "e2e_grouped_i32")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="distinct batches per timed call")
    ap.add_argument("--warmup", type=int, default=3, help="untimed calls of every form before the timed ones")
    ap.add_argument("--batches", type=int, default=200, help="timed batches per form, at least")
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--queries", type=int, default=None)
    ap.add_argument("--negs", type=int, default=None)
    ap.add_argument("--depth", type=int, default=4)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    args.workload = "citation2"          # the workload whose queries share their source
    if args.steps < 1 or args.warmup < 1:
        ap.error("--steps and --warmup must be at least 1")
    return args


def gpu_info(index):
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                        "-i", str(index)], capture_output=True, text=True, check=True)
    name, power, sm = [v.strip() for v in r.stdout.strip().split(",")]
    return {"name": name, "power_limit_w": float(power), "max_sm_mhz": float(sm)}


def h2d_bytes(form, L, bs, K):
    """Bytes of ids one call ships to the device: every batch's pairs, or its targets plus the sources it touches."""
    if form == "e2e_pairs":
        return 16 * L
    if not form.startswith("e2e_grouped"):
        return 0
    w = 4 if form.endswith("i32") else 8
    total = 0
    for lo in range(0, L, bs):
        hi = min(L, lo + bs)
        total += w * ((hi - lo) + (hi - 1) // K + 1 - lo // K)
    return total


def main():
    args = parse()
    import torch.distributed as dist
    import lpformer_b200 as L_
    from lpformer_b200 import _lib, synthetic as S
    from lpformer_b200.evaluate import LinkScoreStream, propagate_replicated

    rank, local_rank, world = B.env_rank()
    if not torch.cuda.is_available():
        raise SystemExit("query_groups_bench.py needs a CUDA device: lpformer_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()
    gpu = gpu_info(local_rank) if rank == 0 else None

    g, negs, _ = B.make_workload(args, rank)
    cfg = g.cfg
    torch.manual_seed(args.seed)
    model = L_.LinkTransformer(S.train_args_of(cfg), g.data_dict(dev), device=dev).to(dev).eval()
    score = L_.mlp_score(model.out_dim, model.out_dim, 1, 2).to(dev).eval()
    X = propagate_replicated(model)
    nq = B.queries_per_step(args, cfg, negs)
    K = 1 + negs
    nlinks = nq * K
    host = np.concatenate([B.make_queries(g, args.workload, nq, negs, seed=1000 + rank * 100003 + s)
                           for s in range(args.warmup, args.warmup + args.steps)], axis=1)
    L = host.shape[1]
    pairs = torch.from_numpy(host)
    src, tgt = pairs[0, ::K].contiguous(), pairs[1].reshape(-1, K).contiguous()
    assert torch.equal(src.repeat_interleave(K), pairs[0]), "every query's links share its source"
    inputs = {
        "dev_pairs": (pairs.to(dev),),
        "dev_grouped_i32": (src.int().to(dev), tgt.int().to(dev)),
        "e2e_pairs": (pairs.pin_memory(),),
        "e2e_grouped_i64": (src.pin_memory(), tgt.pin_memory()),
        "e2e_grouped_i32": (src.int().pin_memory(), tgt.int().pin_memory()),
    }
    out_host = {f: torch.empty(L, dtype=torch.float32).pin_memory() for f in FORMS if f.startswith("e2e")}
    scorer = LinkScoreStream(model, score, X, nlinks, depth=args.depth)

    def run(form):
        a = inputs[form]
        oh = out_host.get(form)
        if len(a) == 1:
            return scorer.score(a[0], out_host=oh)
        return scorer.score_grouped(a[0], a[1], out_host=oh).reshape(-1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):          # plans run eagerly once, then capture their graphs; staging buffers allocated
        for f in FORMS:
            run(f)
    barrier()
    reps = max(1, -(-args.batches // args.steps))
    times = {f: [] for f in FORMS}
    outs = {}
    for r in range(reps):
        order = FORMS[r % len(FORMS):] + FORMS[:r % len(FORMS)]          # rotate: no form always follows the same one
        for f in order:
            barrier()
            if f.startswith("dev"):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                outs[f] = run(f)
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1)
            else:
                t0 = time.perf_counter()
                outs[f] = run(f)
                torch.cuda.synchronize()
                ms = (time.perf_counter() - t0) * 1e3
            times[f].append(ms / args.steps)
    barrier()
    ref = outs["dev_pairs"]
    diffs = {f: float((outs[f] - ref).abs().max()) for f in FORMS}
    host_exact = all(torch.equal(out_host[f], outs[f].cpu()) for f in out_host)
    per = torch.tensor([[sum(times[f]) / reps for f in FORMS] + [diffs[f] for f in FORMS]], dtype=torch.float64,
                       device=dev)
    if world > 1:
        dist.all_reduce(per, op=dist.ReduceOp.MAX)          # the slowest rank, the largest difference
    per = per[0].tolist()
    if rank == 0:
        forms = {}
        for i, f in enumerate(FORMS):
            t = sorted(times[f])
            forms[f] = {"ms_per_step": per[i],
                        "ms_per_step_calls": {"min": t[0], "median": float(np.median(t)), "max": t[-1], "calls": len(t)},
                        "links_per_s": world * nlinks / (per[i] * 1e-3),
                        "h2d_bytes_per_step": h2d_bytes(f, L, nlinks, K) / args.steps}
        line = {
            "tool": "tools/query_groups_bench.py",
            "workload": B.workload_name(args.workload, negs) + (" (scale %g)" % args.scale if args.scale != 1.0 else ""),
            "world_size": world, "gpu": gpu, "queries_per_step": nq, "K": K, "links_per_step": nlinks,
            "steps_per_call": args.steps, "timed_batches_per_form": reps * args.steps, "depth": args.depth,
            "forms": forms,
            "max_abs_diff_vs_dev_pairs": {f: per[len(FORMS) + i] for i, f in enumerate(FORMS)},
            "max_abs_diff": max(per[len(FORMS):]),
            "out_host_equals_device_scores": host_exact,
            "h2d_ratio_pairs_over_grouped_i32": forms["e2e_pairs"]["h2d_bytes_per_step"] /
                                                forms["e2e_grouped_i32"]["h2d_bytes_per_step"],
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
