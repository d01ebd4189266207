#!/usr/bin/env python
"""One training step on bench.py's citation2-shaped graph: one JSON line.

The step is the body of the reference's train/train_model.py:train_epoch at dropout 0 on lpformer_b200's modules:
propagate (the GCN over all 2.93 M nodes + gnn_norm), LinkTransformer.forward on P positive links (train edges) and P
uniformly drawn negatives, mlp_score, the loss -log(pos + 1e-6).mean() - log(1 - neg + 1e-6).mean(), backward and an
Adam step.  The graph is the stored train graph (no per-batch masked adjacency).

Reports ms per step (device events around the whole step, mean and spread over the timed steps), the per-kernel
split (CUDA events around every C-ABI call of one further traced step, summed per entry point; the traced step is not
among the timed ones), peak device memory of a step, and the GPU's name, power limit and max SM clock (read-only
nvidia-smi query in the same run).

With --feat-drop / --gnn-drop / --dropout / --att-drop / --pred-dropout (all 0 by default) the modules train with
those dropouts (the reference's run-script arguments of the same names; --pred-dropout is mlp_score's), and the line
gains a "dropout" field.

  python tools/train_step_bench.py [--links 32768 --steps 5 --warmup 2] [--feat-drop 0.1 --gnn-drop 0.1 ...]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

import bench as B  # noqa: E402


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--links", type=int, default=32768, help="positive links per step (as many negatives)")
    ap.add_argument("--steps", type=int, default=5, help="timed steps")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--seed", type=int, default=0)
    for name in ("feat-drop", "gnn-drop", "dropout", "att-drop", "pred-dropout"):
        ap.add_argument("--" + name, type=float, default=0.0)
    args = ap.parse_args()
    args.workload, args.negs = "citation2", None
    if args.steps < 1 or args.warmup < 1 or args.links < 1:
        ap.error("--steps, --warmup and --links must be at least 1")
    return args


def gpu_info(index):
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                        "-i", str(index)], capture_output=True, text=True, check=True)
    name, power, sm = [v.strip() for v in r.stdout.strip().split(",")]
    return {"name": name, "power_limit_w": float(power), "max_sm_mhz": float(sm)}


def main():
    args = parse()
    import lpformer_b200 as L_
    from lpformer_b200 import _lib, synthetic as S

    if not torch.cuda.is_available():
        raise SystemExit("train_step_bench.py needs a CUDA device: lpformer_b200 has no CPU fallback")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    _lib.load()
    gpu = gpu_info(0)

    g, negs, _ = B.make_workload(args, 0)
    torch.manual_seed(args.seed)
    drops = {"feat_drop": args.feat_drop, "gnn_drop": args.gnn_drop, "dropout": args.dropout, "att_drop": args.att_drop}
    model = L_.LinkTransformer(dict(S.train_args_of(g.cfg), **drops), g.data_dict(dev), device=dev).to(dev).train()
    score = L_.mlp_score(model.out_dim, model.out_dim, 1, 2, dropout=args.pred_dropout).to(dev).train()
    opt = torch.optim.Adam(list(model.parameters()) + list(score.parameters()), lr=1e-3)
    rng = np.random.default_rng(args.seed)
    E = g.edges.shape[1]
    P = args.links

    def batch(step):
        pos = g.edges[:, rng.integers(0, E, P)]
        neg = rng.integers(0, g.n, (2, P))
        return torch.from_numpy(np.concatenate([pos, neg], 1).astype(np.int64)).to(dev)

    def step(links):
        opt.zero_grad(set_to_none=True)
        prob = score(model(links))
        loss = -torch.log(prob[:P] + 1e-6).mean() - torch.log(1 - prob[P:] + 1e-6).mean()
        loss.backward()
        opt.step()
        return loss

    for i in range(args.warmup):
        step(batch(i))
    torch.cuda.synchronize()
    links = [batch(args.warmup + i) for i in range(args.steps + 1)]
    times, losses = [], []
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    for i in range(args.steps):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        loss = step(links[i])
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
        losses.append(float(loss.detach()))
    peak = torch.cuda.max_memory_allocated(dev)

    # per-kernel split of one more step
    tr = _lib.Trace(events=True)
    _lib.TRACE = tr
    torch.cuda.synchronize()
    step(links[-1])
    torch.cuda.synchronize()
    _lib.TRACE = None
    split = {k: {"calls": c, "ms": ms} for k, (c, ms) in sorted(tr.summary().items(), key=lambda kv: -kv[1][1])}
    t = sorted(times)
    line = {
        "tool": "tools/train_step_bench.py",
        "workload": "ogbl-citation2-shaped synthetic graph of bench.py" + (" (scale %g)" % args.scale if args.scale != 1.0 else ""),
        "gpu": gpu, "num_nodes": g.n, "positives": P, "negatives": P, "optimizer": "Adam",
        "ms_per_step": float(np.mean(t)), "ms_per_step_steps": {"min": t[0], "median": float(np.median(t)), "max": t[-1],
                                                                 "steps": len(t)},
        "kernel_ms_per_step": split,
        "kernel_ms_total": float(sum(v["ms"] for v in split.values())),
        "peak_device_memory_gb": peak / 1e9, "resident_before_step_gb": base / 1e9,
        "losses": losses,
    }
    if any(drops.values()) or args.pred_dropout:
        line["dropout"] = dict(drops, pred_dropout=args.pred_dropout)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
