#!/usr/bin/env python
"""Top-k retrieval over all nodes vs materialised scores on the citation2 workload: one JSON line.

For Q sources of bench.py's seeded full-scale citation2 graph (2.93 M nodes; Q = 16: 47 M candidate links per call),
with bench.py's default batch (2,048 queries x 1,001 links = 2,050,048 links per batch), this script times, alternating
the forms call by call:

  topk            LinkScoreStream.top_targets(source, k): every node a candidate, the source left out
  topk_filtered   the same with exclude = the train adjacency and a held-out positive per source (filtered ranks)
  grouped         LinkScoreStream.score_grouped(source, arange(N) per query): the [Q, N] scores materialised

Per form: ms_per_call (mean over the timed calls, device events around the call) with its spread, ms_per_batch and
links_per_s.  Then the fold kernel's own device time per batch (lpf_topk_fold, CUDA events around every call) when
the grouped form's scores are folded batch by batch in the sweep's order, unfiltered and filtered, and its share of
the grouped form's time per batch.  Checks: top_targets' scores against torch.topk of the materialised scores (max
abs difference of the k-th score), and the fraction of returned targets they share.  Also the GPU's name, power limit
and max SM clock (read-only nvidia-smi query in the same run).

  python tools/top_targets_bench.py [--sources 16 --k 100 --calls 5 --warmup 1]
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

FORMS = ("topk", "topk_filtered", "grouped")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sources", type=int, default=16, help="queries per call (each sweeps all N nodes)")
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--calls", type=int, default=5, help="timed calls per form")
    ap.add_argument("--warmup", type=int, default=1, help="untimed calls of every form before the timed ones")
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--depth", type=int, default=4)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    args.workload, args.negs, args.queries = "citation2", None, None     # bench.py's workload and default batch
    if args.calls < 1 or args.warmup < 1 or args.sources < 1:
        ap.error("--calls, --warmup and --sources must be at least 1")
    return args


def gpu_info(index):
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                        "-i", str(index)], capture_output=True, text=True, check=True)
    name, power, sm = [v.strip() for v in r.stdout.strip().split(",")]
    return {"name": name, "power_limit_w": float(power), "max_sm_mhz": float(sm)}


def main():
    args = parse()
    import lpformer_b200 as L_
    from lpformer_b200 import _lib, ops, synthetic as S
    from lpformer_b200.evaluate import LinkScoreStream, propagate_replicated

    if not torch.cuda.is_available():
        raise SystemExit("top_targets_bench.py needs a CUDA device: lpformer_b200 has no CPU fallback")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    _lib.load()
    gpu = gpu_info(0)

    g, negs, _ = B.make_workload(args, 0)
    torch.manual_seed(args.seed)
    model = L_.LinkTransformer(S.train_args_of(g.cfg), g.data_dict(dev), device=dev).to(dev).eval()
    score = L_.mlp_score(model.out_dim, model.out_dim, 1, 2).to(dev).eval()
    X = propagate_replicated(model)
    bs = B.queries_per_step(args, g.cfg, negs) * (1 + negs)
    scorer = LinkScoreStream(model, score, X, bs, depth=args.depth)
    N, Q, k = scorer.num_nodes, args.sources, args.k
    src = torch.from_numpy(g.heldout[0, :Q].copy()).to(dev)
    pos = torch.from_numpy(g.heldout[1, :Q].copy()).to(dev)
    ex = model.get_adj(False, mask=True)
    targets = torch.arange(N, dtype=torch.int32, device=dev).expand(Q, N).contiguous()
    src32 = src.int()

    def run(form):
        if form == "topk":
            return scorer.top_targets(src, k)
        if form == "topk_filtered":
            return scorer.top_targets(src, k, exclude=ex, positive=pos)
        return scorer.score_grouped(src32, targets)

    for _ in range(args.warmup):
        for f in FORMS:
            run(f)
    torch.cuda.synchronize()
    times = {f: [] for f in FORMS}
    outs = {}
    for r in range(args.calls):
        order = FORMS[r % len(FORMS):] + FORMS[:r % len(FORMS)]          # rotate: no form always follows the same one
        for f in order:
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            outs[f] = run(f)
            e1.record()
            torch.cuda.synchronize()
            times[f].append(e0.elapsed_time(e1))
    L = Q * N
    nb = -(-L // bs)

    # the fold alone: the materialised scores folded batch by batch in the sweep's order, CUDA events around each call
    S_flat = outs["grouped"].reshape(-1)
    pos_score = scorer.score(torch.stack((src, pos)))
    fold_ms = {}
    for name, kw in (("topk", {}), ("topk_filtered", dict(exclude=ex, positive=pos))):
        ws = ops.topk_fold_workspace(bs, k, N, dev)
        per_batch = []
        for _ in range(args.calls):
            top_key = torch.full((Q, k), float("-inf"), device=dev)
            top_id = torch.full((Q, k), -1, dtype=torch.int32, device=dev)
            cnt = torch.zeros((2, Q), dtype=torch.int64, device=dev)
            extra = {}
            if "positive" in kw:
                extra = dict(positive=pos, pos_score=pos_score, cnt_ge=cnt[0], cnt_gt=cnt[1])
            evs = []
            for lo in range(0, L, bs):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                ops.topk_fold(S_flat[lo:lo + bs], lo, src, N, k, top_key, top_id, ws, exclude=kw.get("exclude"), **extra)
                b.record()
                evs.append((a, b))
            torch.cuda.synchronize()
            per_batch += [a.elapsed_time(b) for a, b in evs]
        fold_ms[name] = {"mean": float(np.mean(per_batch)), "median": float(np.median(per_batch)),
                         "max": float(np.max(per_batch)), "batches": len(per_batch)}

    # checks against the materialised scores
    Sm = outs["grouped"].clone()
    Sm[torch.arange(Q, device=dev), src.long()] = float("-inf")
    ref_v, ref_i = torch.topk(Sm, k, dim=1)
    got = outs["topk"]
    kth_diff = float((got.scores[:, -1] - ref_v[:, -1]).abs().max())
    shared = float(np.mean([len(set(got.targets[q].tolist()) & set(ref_i[q].tolist())) / k for q in range(Q)]))

    forms = {}
    for f in FORMS:
        t = sorted(times[f])
        mean = float(np.mean(t))
        forms[f] = {"ms_per_call": mean, "ms_per_call_calls": {"min": t[0], "median": float(np.median(t)),
                                                               "max": t[-1], "calls": len(t)},
                    "ms_per_batch": mean / nb, "links_per_s": L / (mean * 1e-3)}
    step = forms["grouped"]["ms_per_batch"]
    line = {
        "tool": "tools/top_targets_bench.py",
        "workload": B.workload_name(args.workload, negs) + (" (scale %g)" % args.scale if args.scale != 1.0 else ""),
        "gpu": gpu, "num_nodes": N, "queries": Q, "k": k, "links_per_call": L, "batch": bs, "batches_per_call": nb,
        "depth": args.depth, "forms": forms,
        "topk_over_grouped": forms["topk"]["ms_per_call"] / forms["grouped"]["ms_per_call"],
        "topk_filtered_over_grouped": forms["topk_filtered"]["ms_per_call"] / forms["grouped"]["ms_per_call"],
        "fold_ms_per_batch": fold_ms,
        "fold_share_of_grouped_batch": {n: v["mean"] / step for n, v in fold_ms.items()},
        "kth_score_max_abs_diff_vs_torch_topk": kth_diff,
        "targets_shared_with_torch_topk": shared,
        "filtered_mean_rank": float(outs["topk_filtered"].rank.mean()),
    }
    print(json.dumps(line))


if __name__ == "__main__":
    main()
