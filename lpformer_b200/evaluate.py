"""Eval-side drivers around LinkTransformer: pipelined batch scoring, ranking metrics on the device, link-sharded
multi-GPU scoring.

Links are independent units, so candidate links are sharded across ranks with NO per-batch
collective.  The only exchange is per eval: the last GCN layer (+ gnn_norm + the K/V
projection) is computed for a row shard on each rank and the node tables [X | KV] are
replicated by ONE all-gather over NCCL/NVLink (SURVEY.md §8e).
"""
from __future__ import annotations

from collections import namedtuple

import torch
import torch.distributed as dist

from . import _lib, ops
from .graph import csr_from_sparse
from .plan import ScorePlan

TopTargets = namedtuple("TopTargets", "scores targets rank")
TopTargets.__doc__ = """LinkScoreStream.top_targets / top_targets_sharded: scores fp32 [Q, k] and targets int64 [Q, k] of every
query's k best candidates (score descending, then target id ascending; (-inf, -1) where a query has fewer than k
candidates), rank fp32 [Q] of the positives among the filtered candidates (None without positives)."""


@torch.no_grad()
def propagate_replicated(model, test_set=False, group=None):
    """X_node [N, dim] on every rank, with the K/V tables of all attention layers primed.

    world_size 1: plain model.propagate().  Otherwise EVERY GCN layer is row-sharded: a rank applies the layer's Linear
    to its own rows, the ranks all-gather the [N/W, d] products (the SpMM gathers rows of any node), and the fused
    layer launch (SpMM + bias + LayerNorm + ReLU + residual; for the last layer also gnn_norm) runs for the rank's rows
    only; the K/V projections follow on those rows and ONE all_gather_into_tensor of the packed [X | KV_0 | ...] rows
    replicates the result.  Per eval: L all-gathers of [N, d] and one of [N, d + sum HC], no collective per batch."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        X = model.propagate(test_set=test_set)
        model._get_kv(X)
        return X
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    dev = model._dev()
    adj = model.get_adj(test_set)
    n, d = adj.n, model.dim
    x = model.data["x"]
    if "emb" in model.data:
        x = model.data["emb"](x)
    x = x.detach().to(dev, torch.float32)
    gcn = model.node_encoder.gnn_encoder
    convs = list(gcn.convs)
    per = (n + world - 1) // world
    r0 = min(n, rank * per)
    rows = min(n, r0 + per) - r0
    x_own = x[r0:r0 + rows].contiguous()                 # this rank's rows of the layer input
    for i, conv in enumerate(convs):
        last = i == len(convs) - 1
        ln = gcn.lns[i] if gcn.lns is not None else None
        width = conv.bias.numel()
        xw_own = torch.zeros((per, width), dtype=torch.float32, device=dev)
        if rows > 0:
            ops.linear(x_own, conv.lin.weight, out=xw_own[:rows])
        xw = torch.empty((per * world, width), dtype=torch.float32, device=dev)
        dist.all_gather_into_tensor(xw, xw_own, group=group)
        res = x_own if (gcn.residual and x_own.shape[-1] == width) else None
        y_own = torch.empty((max(rows, 1), width), dtype=torch.float32, device=dev)
        if rows > 0:
            ops.gcn_layer(adj, xw[:n], conv.bias, ln=None if ln is None else (ln.weight, ln.bias), relu=gcn.relu, residual=res,
                          ln2=(model.gnn_norm.weight, model.gnn_norm.bias) if last else None, out=y_own, row0=r0, rows=rows,
                          local=True)
        x_own = y_own[:rows]
    widths = [d] + [layer.att.heads * layer.att.out_channels for layer in model.att_layers]
    packed = torch.zeros((per, sum(widths)), dtype=torch.float32, device=dev)
    if rows > 0:
        packed[:rows, :d].copy_(x_own)
        xs = packed[:rows, :d]
        c0 = d
        for layer, w in zip(model.att_layers, widths[1:]):
            ops.linear(xs, layer.att.lin_r.weight[:, :d], out=packed[:rows, c0:c0 + w])
            c0 += w
    full = torch.empty((per * world, sum(widths)), dtype=torch.float32, device=dev)
    dist.all_gather_into_tensor(full, packed, group=group)          # the one collective that replicates the tables
    full = full[:n]
    X = full[:, :d]
    kvs, c0 = [], d
    for w in widths[1:]:
        kvs.append(full[:, c0:c0 + w])
        c0 += w
    model._prime_kv(X, kvs)
    return X


def shard_queries(num_queries, rank, world):
    """Contiguous query-group shard [lo, hi) of this rank (a citation2 source's 1000 negatives stay together)."""
    per = (num_queries + world - 1) // world
    lo = min(num_queries, rank * per)
    return lo, min(num_queries, lo + per)


def shard_bounds(num_queries, world, cost=None):
    """The world + 1 boundaries of the contiguous query-group shards.  cost (optional, one non-negative number per group):
    the shards are cut so that every rank gets the same share of the total COST instead of the same number of groups —
    a link costs what its two rows weigh (SURVEY 8(e): "balance by sum(deg + nP), not link count"), and a few hub
    sources can double one rank's share.  Deterministic: every rank computes the same cuts from the same links."""
    if cost is None or num_queries == 0 or world == 1:
        return [shard_queries(num_queries, r, world)[0] for r in range(world)] + [num_queries]
    csum = torch.cumsum(torch.as_tensor(cost, dtype=torch.float64).reshape(-1).cpu(), 0)
    total = float(csum[-1])
    if not total > 0.0:
        return [shard_queries(num_queries, r, world)[0] for r in range(world)] + [num_queries]
    targets = torch.tensor([total * r / world for r in range(1, world)], dtype=torch.float64)
    cuts = torch.searchsorted(csum, targets, right=False).tolist()      # first group whose running cost reaches the target
    bounds = [0] + [min(num_queries, int(c) + 1) for c in cuts] + [num_queries]
    for i in range(1, len(bounds)):                                       # (monotone even with zero-cost groups)
        bounds[i] = max(bounds[i], bounds[i - 1])
    return bounds


def _row_bytes(model, test_set):
    """float64 [N]: the bytes of a node's adjacency and PPR rows the selection reads (4 deg + 8 nP)."""
    adj, ppr = model.get_adj(test_set, mask=True), model.get_ppr(test_set)
    return (4 * (adj.rowptr[1:] - adj.rowptr[:-1]) + 8 * (ppr.rowptr[1:] - ppr.rowptr[:-1])).to(torch.float64)


def query_group_cost(model, source, targets, test_set=False):
    """link_group_cost of the expanded links of query groups (source [Q], targets [Q, K]), from the grouped form: the
    source's row once, every target's row, 48 bytes per link."""
    row = _row_bytes(model, test_set)
    dev = row.device
    return row[source.to(dev).long()] + row[targets.to(dev).long()].sum(1) + 48.0 * targets.shape[1]


def link_group_cost(model, links, group_size, test_set=False):
    """Cost of every group of `group_size` consecutive links: 4 deg + 8 nP (+ 48) bytes of both endpoints' rows, the
    shared source of a citation2-style group counted once (the algorithmic bytes of the selection, SURVEY 8(d))."""
    row = _row_bytes(model, test_set)
    dev = row.device
    lk = links.to(dev)
    ng = lk.shape[1] // group_size
    a = lk[0, :ng * group_size].reshape(ng, group_size)
    b = lk[1, :ng * group_size].reshape(ng, group_size)
    same_src = bool((a == a[:, :1]).all()) if ng > 0 else False
    cost_a = row[a[:, 0]] if same_src else row[a].sum(1)
    return cost_a + row[b].sum(1) + 48.0 * group_size


@torch.no_grad()
def score_links_sharded(model, score_func, links, X, test_set=False, group=None, group_size=1, batch_size=None,
                        balance=True):
    """Scores `links` [2, L] (L a multiple of group_size) with link groups sharded over the ranks of
    `group`; returns the full [L] probabilities on every rank (one all_gather of fp32 scores at the end).
    balance: cut the shards by the weight of the links' rows (shard_bounds / link_group_cost) instead of by count."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    dev = model._dev()
    L = links.shape[1]
    ngroups = L // group_size
    cost = link_group_cost(model, links, group_size, test_set) if (balance and world > 1 and hasattr(model, "get_adj")) else None
    bounds = shard_bounds(ngroups, world, cost)
    lo, hi = bounds[rank], bounds[rank + 1]
    mine = links[:, lo * group_size:hi * group_size].to(dev)
    bs = batch_size or max(1, mine.shape[1])
    outs = [model.score_links(mine[:, s:s + bs], X, score_func, test_set=test_set) for s in range(0, mine.shape[1], bs)]
    local = torch.cat(outs) if outs else torch.empty(0, device=dev)
    if world == 1:
        return local
    per = max(1, max(bounds[r + 1] - bounds[r] for r in range(world)) * group_size)
    pad = torch.zeros(per, dtype=torch.float32, device=dev)
    pad[:local.numel()] = local
    full = torch.empty(per * world, dtype=torch.float32, device=dev)
    dist.all_gather_into_tensor(full, pad, group=group)
    pieces = []
    for r in range(world):
        pieces.append(full[r * per:r * per + (bounds[r + 1] - bounds[r]) * group_size])
    return torch.cat(pieces)


@torch.no_grad()
def score_queries_sharded(model, score_func, source, targets, X, test_set=False, group=None, batch_size=None,
                          balance=True):
    """score_links_sharded for query groups (source [Q], targets [Q, K], int32 or int64 alike): the queries are sharded
    over the ranks of `group`, every rank ships and scores only its own (model.score_queries, batch_size links per call
    rounded down to whole queries), and one all_gather of fp32 scores returns the full [Q, K] on every rank.
    balance: cut the shards by the weight of the links' rows (shard_bounds / query_group_cost) instead of by count."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    dev = model._dev()
    source, targets = ops.query_groups(source, targets)
    Q, K = targets.shape
    cost = query_group_cost(model, source, targets, test_set) if (balance and world > 1 and hasattr(model, "get_adj")) else None
    bounds = shard_bounds(Q, world, cost)
    lo, hi = bounds[rank], bounds[rank + 1]
    src, tgt = source[lo:hi].to(dev), targets[lo:hi].to(dev)
    qb = max(1, (batch_size or max(1, (hi - lo) * K)) // max(1, K))
    outs = [model.score_queries(src[s:s + qb], tgt[s:s + qb], X, score_func, test_set=test_set) for s in range(0, hi - lo, qb)]
    local = torch.cat(outs) if outs else torch.empty((0, K), device=dev)
    if world == 1:
        return local
    per = max(1, max(bounds[r + 1] - bounds[r] for r in range(world)) * K)
    pad = torch.zeros(per, dtype=torch.float32, device=dev)
    pad[:local.numel()] = local.reshape(-1)
    full = torch.empty(per * world, dtype=torch.float32, device=dev)
    dist.all_gather_into_tensor(full, pad, group=group)
    pieces = [full[r * per:r * per + (bounds[r + 1] - bounds[r]) * K] for r in range(world)]
    return torch.cat(pieces).view(Q, K)


@torch.no_grad()
def top_targets_sharded(model, score_func, source, X, k, exclude=None, positive=None, test_set=False, group=None,
                        batch_size=None, stream=None):
    """LinkScoreStream.top_targets with the queries sharded over the ranks of `group`: every query costs one sweep of
    all N nodes, so the shards are cut by count (shard_bounds); each rank runs its own stream (`stream`, or one of
    batch_size links, default 2^21) on its queries, and ONE all_gather of the padded [Q_r, k] results (plus the ranks)
    returns the full TopTargets on every rank."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    src = torch.as_tensor(source)
    Q = src.shape[0]
    bounds = shard_bounds(Q, world)
    lo, hi = bounds[rank], bounds[rank + 1]
    st = stream if stream is not None else LinkScoreStream(model, score_func, X, batch_size or (1 << 21),
                                                           test_set=test_set)
    mine = st.top_targets(src[lo:hi], k, exclude=exclude,
                          positive=None if positive is None else torch.as_tensor(positive)[lo:hi])
    if world == 1:
        return mine
    # one float64 row per query: k scores, k target ids and the rank (all exact in float64)
    per = max(1, max(bounds[r + 1] - bounds[r] for r in range(world)))
    w = 2 * k + (positive is not None)
    pad = torch.zeros((per, w), dtype=torch.float64, device=mine.scores.device)
    pad[:hi - lo, :k] = mine.scores
    pad[:hi - lo, k:2 * k] = mine.targets.to(torch.float64)
    if positive is not None:
        pad[:hi - lo, 2 * k] = mine.rank
    full = torch.empty((per * world, w), dtype=torch.float64, device=pad.device)
    dist.all_gather_into_tensor(full, pad, group=group)
    rows = torch.cat([full[r * per:r * per + bounds[r + 1] - bounds[r]] for r in range(world)])
    return TopTargets(rows[:, :k].float(), rows[:, k:2 * k].long(), rows[:, 2 * k].float() if positive is not None else None)


class _Input:
    """What the batch loop does with a batch's scores: by default they go into the [L] output at their flat position."""
    out = None

    def alloc(self):
        self.out = torch.empty(self.L, dtype=torch.float32, device=self.s.dev)
        return self.out

    def take(self, prob, lo, P=None):
        """prob: the scores of flat positions [lo, lo + prob.numel()), on the current stream; P: the plan that produced
        them (None: scored outside the plans)."""
        self.out[lo:lo + prob.numel()].copy_(prob, non_blocking=True)


class _LinkPairs(_Input):
    """Input of LinkScoreStream.score: int64 link pairs [2, L], staged as they are."""

    def __init__(self, stream, links):
        self.s, self.lk, self.L, self.on_host = stream, links, links.shape[1], not links.is_cuda

    def stage(self, G):
        s = self.s
        if s._stage is None or s._stage[0].shape[1] != G * s.bs:
            s._stage = [torch.empty((2, G * s.bs), dtype=torch.int64, device=s.dev) for _ in range(2)]
        return s._stage

    def h2d(self, slot, j, k):
        # row by row: a strided two-row host slice would go through a slow pitched copy (15 vs 48 GB/s measured)
        bs, lo = self.s.bs, k * self.s.bs
        slot[0, j * bs:(j + 1) * bs].copy_(self.lk[0, lo:lo + bs], non_blocking=True)
        slot[1, j * bs:(j + 1) * bs].copy_(self.lk[1, lo:lo + bs], non_blocking=True)

    def submit(self, P, slot, j, k):
        bs = self.s.bs
        P.submit(slot[:, j * bs:(j + 1) * bs] if slot is not None else self.lk[:, k * bs:(k + 1) * bs])

    def links(self, lo, hi):
        return self.lk[:, lo:hi]

    def begin(self):
        pass

    def check(self, plan_bad, expanded):
        pass


class _QueryGroups(_Input):
    """Input of LinkScoreStream.score_grouped: source [Q] and targets [Q, K] (int32 or int64), flat link i = q K + j.  A
    batch is staged as its targets plus the sources it touches and expanded into the plan's links buffer on the device.
    Out-of-range ids are flagged in word 5 of the plan's header (no selection launch writes it; collect() reads the
    header back every batch anyway) or, for batches expanded outside a plan, in the stream's own word."""
    what = "query groups hold a node id"

    def __init__(self, stream, source, targets):
        self.s, self.src, self.K = stream, source, targets.shape[1]
        self.tgt = targets.reshape(-1)
        self.L, self.on_host = self.tgt.numel(), not targets.is_cuda
        self.S = stream.bs // self.K + 2          # sources a batch of bs links touches at most

    def stage(self, G):
        s, dt = self.s, self.tgt.dtype          # (kept per id width: callers may alternate int32 and int64 groups)
        st = s._gstage.get(dt)
        if st is None or st[0][0].numel() != G * s.bs or st[0][1].numel() != G * self.S:
            st = s._gstage[dt] = [(torch.empty(G * s.bs, dtype=dt, device=s.dev),
                                   torch.empty(G * self.S, dtype=dt, device=s.dev)) for _ in range(2)]
        return st

    def _span(self, lo, hi):
        return lo // self.K, (hi - 1) // self.K + 1

    def h2d(self, slot, j, k):
        bs, S, lo = self.s.bs, self.S, k * self.s.bs
        q0, q1 = self._span(lo, lo + bs)
        slot[0][j * bs:(j + 1) * bs].copy_(self.tgt[lo:lo + bs], non_blocking=True)
        slot[1][j * S:j * S + q1 - q0].copy_(self.src[q0:q1], non_blocking=True)

    def submit(self, P, slot, j, k):
        bs, lo = self.s.bs, k * self.s.bs
        if slot is not None:
            src, tgt = slot[1][j * self.S:], slot[0][j * bs:]
        else:
            src, tgt = self.src[lo // self.K:], self.tgt[lo:]
        ops.expand_query_links(src, tgt, self.K, lo % self.K, bs, self.s.num_nodes, P.links, P.hdr[5:6])
        P.submit(None)

    def links(self, lo, hi):
        """The int64 links [2, hi - lo] of a flat range, expanded on the device (ragged tail, overflow redo)."""
        q0, q1 = self._span(lo, hi)
        dev = self.s.dev
        out = torch.empty((2, hi - lo), dtype=torch.int64, device=dev)
        if hi > lo:
            ops.expand_query_links(self.src[q0:q1].to(dev), self.tgt[lo:hi].to(dev), self.K, lo - q0 * self.K, hi - lo,
                                   self.s.num_nodes, out, self.s._bad)
        return out

    def begin(self):
        """Resets the flags once per call (on the caller's stream, which every plan stream then waits for)."""
        s = self.s
        if s._bad is None:
            s._bad = torch.zeros(1, dtype=torch.int64, device=s.dev)
        s._bad.zero_()
        for P in s.plans or []:
            P.hdr[5:6].zero_()

    def check(self, plan_bad, expanded):
        """Raises once the call is drained if a plan or an expansion outside the plans met an out-of-range id (the
        stream's word is read only when such an expansion ran, i.e. after a host round trip the call makes anyway)."""
        if plan_bad or (expanded and int(self.s._bad.item())):
            raise _lib.LpfError(f"{self.what} outside [0, {self.s.num_nodes})")


class _SourceSweep(_QueryGroups):
    """Input of LinkScoreStream.top_targets: the query groups (source[q], every node j < N), flat link i = q N + j,
    never materialised.  Each batch is expanded on the device (lpf_expand_source_sweep) and its scores are folded into
    per-query top-k state and rank counters (lpf_topk_fold) instead of being kept: no [L] output exists."""
    what = "sources hold a node id"

    def __init__(self, stream, source, k, exclude, positive, pos_score):
        self.s, self.src, self.K = stream, source, stream.num_nodes
        self.L, self.on_host = source.numel() * self.K, False
        Q, dev = source.numel(), stream.dev
        self.k, self.exclude, self.positive, self.pos_score = k, exclude, positive, pos_score
        self.top_key = torch.full((Q, k), float("-inf"), dtype=torch.float32, device=dev)
        self.top_id = torch.full((Q, k), -1, dtype=torch.int32, device=dev)
        self.cnt = torch.zeros((2, Q), dtype=torch.int64, device=dev) if positive is not None else None
        self.ws = ops.topk_fold_workspace(stream.bs, k, self.K, dev)

    def submit(self, P, slot, j, k):
        bs, lo = self.s.bs, k * self.s.bs
        ops.expand_source_sweep(self.src[lo // self.K:], self.K, lo % self.K, bs, self.s.num_nodes, P.links, P.hdr[5:6])
        P.submit(None)

    def links(self, lo, hi):
        """The int64 links [2, hi - lo] of a flat range, expanded on the device (ragged tail, overflow redo)."""
        q0 = lo // self.K
        out = torch.empty((2, hi - lo), dtype=torch.int64, device=self.s.dev)
        if hi > lo:
            ops.expand_source_sweep(self.src[q0:], self.K, lo - q0 * self.K, hi - lo, self.s.num_nodes, out, self.s._bad)
        return out

    def alloc(self):
        return None

    def take(self, prob, lo, P=None):
        """Folds the scores.  The folds of one call update the same state, so they run one after another on the
        stream's fold stream: a plan's batch is folded there once its launch is through, with the plan's overflow word
        as the skip word (an overflowed batch is folded when it is re-scored, in any order: the fold's result does not
        depend on it), and the plan's next batch waits until the fold has read the plan's scores.  Scores produced
        outside the plans are folded on the current stream, after every plan stream has drained."""
        if P is None:
            self._fold(prob, lo, None)
            return
        cur, fs = torch.cuda.current_stream(self.s.dev), self.s.fold_stream
        fs.wait_stream(cur)
        with torch.cuda.stream(fs):
            self._fold(prob, lo, P.hdr[4:5])
        cur.wait_stream(fs)

    def _fold(self, prob, lo, skip):
        c = self.cnt
        ops.topk_fold(prob, lo, self.src, self.K, self.k, self.top_key, self.top_id, self.ws, exclude=self.exclude,
                      positive=self.positive, pos_score=self.pos_score, cnt_ge=None if c is None else c[0],
                      cnt_gt=None if c is None else c[1], skip=skip)


class LinkScoreStream:
    """The batch loop of the reference's eval drivers (train/testing.py:25-32, 36-43, 107-117: for every batch
    `elementwise_lin` -> `calc_pairwise` -> `score_func` -> `.cpu()`), pipelined.

    The reference synchronises with the host once per batch (`.cpu()`); `LinkTransformer.score_links` still reads
    one 64-byte header per batch (the pair-pool overflow flag).  Here `depth` execution plans (plan.py) are kept in
    flight: batch k+1 is launched before the header of batch k is looked at, host-resident links travel on a copy
    stream next to the compute of the previous batch, and a batch whose pair pool overflowed (detected `depth`
    batches later) is re-scored through the host-sized path at the end — so the scores are exactly those of
    `score_links`, without a GPU idle gap per batch.
    """

    def __init__(self, model, score_func, X_node, batch_size, test_set=False, depth=4, return_logits=False):
        self.model, self.score_func, self.bs = model, score_func, int(batch_size)
        self.test_set, self.logits = bool(test_set), bool(return_logits)
        self.X = model._check_x(X_node)
        self.dev = self.X.device
        consts = model._head_consts(score_func, self.X)
        adj, ppr = model.get_adj(test_set, mask=True), model.get_ppr(test_set)
        algo = ops.pick_select_algo(adj, ppr, model.thresh_1hop, model.thresh_non1hop, model.mask)
        self.plans = None
        if consts is not None and algo != _lib.ALGO_GENERIC and model.use_plans and self.bs > 0:
            kv = model._get_kv(self.X)[0]
            self.plans = [ScorePlan(model, score_func, consts, self.X, kv, self.bs, test_set, return_logits,
                                    use_graph=model.use_graphs) for _ in range(max(1, int(depth)))]
        self.copy_stream = torch.cuda.Stream(device=self.dev)
        self.out_stream = torch.cuda.Stream(device=self.dev)     # scores to the host: the other direction of the link
        # every plan launches on a stream of its own: the latency-bound tail of one batch (hub sources, heavy links,
        # the non-empty links) overlaps the bandwidth-bound head of the next
        self.streams = [torch.cuda.Stream(device=self.dev) for _ in (self.plans or [])]
        self.fold_stream = torch.cuda.Stream(device=self.dev)     # top_targets: the folds, one after another
        self._stage = None
        self._gstage = {}
        self._bad = None
        self.num_nodes = model._id_bound(self.X, test_set)
        self.batches = 0

    def _sequential(self, inp):
        for s in range(0, inp.L, max(1, self.bs)):
            b = inp.links(s, min(inp.L, s + self.bs))
            inp.take(self.model.score_links(b, self.X, self.score_func, test_set=self.test_set,
                                            return_logits=self.logits), s)

    @torch.no_grad()
    def score(self, links, out_host=None, group=4):
        """Scores links [2, L] (int64; a device tensor or pinned host memory).  Returns the [L] scores on the
        device; with `out_host` (a pinned fp32 [L] tensor) the scores are also copied to the host as they are
        produced (the reference's per-batch `.cpu()`), complete when the call returns.  Host-resident links and the
        scores travel in groups of `group` batches on a copy stream: the links of group g+1 are on their way while
        group g is scored."""
        return self._score(_LinkPairs(self, links), out_host, group)

    @torch.no_grad()
    def score_grouped(self, source, targets, out_host=None, group=4):
        """score() for query groups: source [Q] and targets [Q, K] (both int32 or both int64; device tensors or pinned
        host memory) stand for the Q*K links (source[q], targets[q, j]) in that flat order (the reference's citation2
        eval input, train/testing.py:14-27).  Returns the [Q, K] scores on the device; out_host: a pinned fp32 [Q*K]
        tensor, as in score().

        The batches are those score() forms on the expanded links — contiguous ranges of batch_size links, which may
        straddle queries — run in the same order through the same plans.  Host-resident groups ship 4 or 8 bytes per
        link (the target) plus the few sources a batch touches, instead of 16 bytes per link; each batch is expanded
        into its plan's links buffer on the device (lpf_expand_query_links).  A node id outside [0, num_nodes) raises
        LpfError once the call has drained its streams; the stream stays usable."""
        source, targets = ops.query_groups(source, targets)
        Q, K = targets.shape
        if Q * K == 0:
            return torch.empty((Q, K), dtype=torch.float32, device=self.dev)
        return self._score(_QueryGroups(self, source, targets), out_host, group).view(Q, K)

    @torch.no_grad()
    def top_targets(self, source, k, exclude=None, positive=None):
        """Top-k retrieval over every node: for each source[q] the k targets with the highest scores among all N nodes
        (N = the stream's node-id bound) except the source itself and, with `exclude`, the source's row of that
        adjacency (anything graph.csr_from_sparse accepts; a filtered evaluation passes model.get_adj(False,
        mask=True)).  The scores are this stream's: probabilities, or logits with return_logits.

        positive [Q] (optional): rank of each positive among the same filtered candidates (the positive left out),
        1 + (#(score >= s_pos) + #(score > s_pos)) / 2 — get_ranking_list's convention with those candidates as the
        negatives — where s_pos is the positive link's score from score().

        source / positive: int32 or int64, on the device or in host memory.  Returns TopTargets(scores fp32 [Q, k],
        targets int64 [Q, k], rank fp32 [Q] or None) on the device.  The Q x N candidate links run through the same
        batches and plans as score() — expanded on the device batch by batch and folded there into a fixed [Q, k]
        state (lpf_topk_fold) — and are never materialised.  A source or positive outside [0, N), or a positive equal to
        its source, raises LpfError."""
        src = torch.as_tensor(source)
        if src.dim() != 1 or src.dtype not in (torch.int32, torch.int64):
            raise ValueError(f"source must be a 1-D int32 or int64 tensor; got {src.dtype} {list(src.shape)}")
        k = int(k)
        if not 1 <= k <= 1024:
            raise ValueError(f"k must be in [1, 1024]; got {k}")
        if self.bs < 1:
            raise ValueError("top_targets needs a batch size >= 1")
        src = src.to(self.dev).contiguous()
        Q, N = src.numel(), self.num_nodes
        if Q > 0 and bool(((src < 0) | (src >= N)).any()):
            raise _lib.LpfError(f"sources hold a node id outside [0, {N})")
        pos = pos_score = None
        if positive is not None:
            pos = torch.as_tensor(positive)
            if pos.shape != src.shape or pos.dtype not in (torch.int32, torch.int64):
                raise ValueError(f"positive must be int32 or int64 [{Q}]; got {pos.dtype} {list(pos.shape)}")
            pos = pos.to(self.dev, src.dtype).contiguous()
            if Q > 0 and bool(((pos < 0) | (pos >= N) | (pos == src)).any()):
                raise _lib.LpfError(f"positives must be node ids in [0, {N}) other than their source")
        if Q == 0:
            return TopTargets(torch.empty((0, k), dtype=torch.float32, device=self.dev),
                              torch.empty((0, k), dtype=torch.int64, device=self.dev),
                              None if pos is None else torch.empty(0, dtype=torch.float32, device=self.dev))
        if pos is not None:
            pos_score = self.score(torch.stack((src.long(), pos.long())))
        ex = None if exclude is None else csr_from_sparse(exclude, device=self.dev, mask=True)
        inp = _SourceSweep(self, src, k, ex, pos, pos_score)
        self._score(inp, None, 4)
        rank = None if pos is None else 0.5 * (inp.cnt[0] + inp.cnt[1]).to(torch.float32) + 1
        return TopTargets(inp.top_key, inp.top_id.long(), rank)

    def _score(self, inp, out_host, group):
        """The pipelined batch loop over the links of `inp` (_LinkPairs, _QueryGroups or _SourceSweep: how a batch is
        staged, how it fills a plan's links buffer and what becomes of its scores).  Returns the [L] scores (None for
        an input that keeps none)."""
        L = inp.L
        out_dev = inp.alloc()
        main = torch.cuda.current_stream(self.dev)
        inp.begin()
        if self.plans is None:
            self._sequential(inp)
            if out_host is not None:
                out_host.copy_(out_dev)
            inp.check(False, True)
            return out_dev
        bs, depth = self.bs, len(self.plans)
        nb = L // bs
        on_host = inp.on_host
        G = max(int(group), depth)
        cs = self.copy_stream
        stage = inp.stage(G) if on_host else None
        ev_in = [[torch.cuda.Event() for _ in range(G)] for _ in range(2)]     # [slot][batch of the group]: its links are in
        ev_free = [torch.cuda.Event(), torch.cuda.Event()]

        def h2d(g):          # links of the group that starts at batch g -> staging slot, on the copy stream
            slot = (g // G) % 2
            with torch.cuda.stream(cs):
                # (the copy stream has already waited for the plans to take the slot's previous links: ev_free)
                # batch by batch, each announced on its own: the first batch of a call starts after ITS links have
                # arrived, not after the whole group's
                for j in range(min(G, nb - g)):
                    inp.h2d(stage[slot], j, g + j)
                    ev_in[slot][j].record(cs)

        pending = [None] * depth
        redo = []
        ev_start = torch.cuda.Event()
        ev_start.record(main)                 # `links` / `out_dev` are ready in the caller's stream order
        for st in self.streams:
            st.wait_event(ev_start)
        if on_host and nb > 0:
            h2d(0)
        for g in range(0, nb, G):
            kb = min(G, nb - g)
            slot = (g // G) % 2
            if on_host and g + G < nb:
                h2d(g + G)
            for j in range(kb):
                k = g + j
                P, st = self.plans[k % depth], self.streams[k % depth]
                if pending[k % depth] is not None and P.collect():
                    redo.append(pending[k % depth])
                with torch.cuda.stream(st):
                    if on_host:
                        st.wait_event(ev_in[slot][j])
                    inp.submit(P, stage[slot] if on_host else None, j, k)
                    inp.take(P.prob, k * bs, P)
                pending[k % depth] = k
                self.batches += 1
            if on_host or out_host is not None:
                # the group is through once every plan stream has passed this point
                # (the links come in on one stream and the scores leave on another: PCIe is full duplex, and on one
                # stream the 4 bytes per link going out would queue behind the 16 coming in)
                for st in self.streams:
                    e = torch.cuda.Event()
                    e.record(st)
                    if on_host:
                        cs.wait_event(e)
                    if out_host is not None:
                        self.out_stream.wait_event(e)
                if on_host:
                    ev_free[slot].record(cs)
                if out_host is not None:
                    with torch.cuda.stream(self.out_stream):
                        out_host[g * bs:(g + kb) * bs].copy_(out_dev[g * bs:(g + kb) * bs], non_blocking=True)
        for j, k in enumerate(pending):
            if k is not None and self.plans[j].collect():
                redo.append(k)
        plan_bad = any(self.plans[j].last[5] for j, k in enumerate(pending) if k is not None)
        if nb * bs < L:
            redo.append(nb)        # the ragged tail goes through score_links
        for st in self.streams:
            st.synchronize()
        cs.synchronize()
        self.out_stream.synchronize()
        if redo:
            use = self.model.use_plans
            self.model.use_plans = False      # host-sized two-pass path: no pools to overflow
            try:
                for k in redo:
                    lk = inp.links(k * bs, min(L, (k + 1) * bs))
                    pr = self.model.score_links(lk.to(self.dev), self.X, self.score_func, test_set=self.test_set,
                                                return_logits=self.logits)
                    inp.take(pr, k * bs)
                    if out_host is not None:
                        out_host[k * bs:k * bs + pr.numel()].copy_(pr)
            finally:
                self.model.use_plans = use
            full = [k for k in redo if k < nb]
            if full:                          # larger pools for the batches to come: grown until a batch that overflowed fits
                probe = inp.links(full[0] * bs, (full[0] + 1) * bs).to(self.dev)
                while True:
                    for P in self.plans:
                        P.grow()
                    if self.plans[0].cap >= 64 * bs or not self.plans[0].run(probe)[1]:
                        break
            main.synchronize()
        inp.check(plan_bad, bool(redo))
        return out_dev


# ------------------------------------------------------------------------------------------------------------
# Ranking metrics on the device (reference train/evaluation.py).  Predictions stay where the scoring left them;
# every result dict costs ONE host read.
# ------------------------------------------------------------------------------------------------------------
@torch.no_grad()
def get_ranking_list(y_pred_pos, y_pred_neg):
    """reference train/evaluation.py:75-90: rank of every positive among ITS negatives (y_pred_neg [P, K]) or among a
    shared list (y_pred_neg [M] / [1, M]), mean of the optimistic and the pessimistic rank."""
    y_pred_pos = y_pred_pos.reshape(-1, 1)
    if y_pred_neg.dim() == 1:
        y_pred_neg = y_pred_neg.reshape(1, -1)
    optimistic = (y_pred_neg >= y_pred_pos).sum(dim=1)
    pessimistic = (y_pred_neg > y_pred_pos).sum(dim=1)
    return 0.5 * (optimistic + pessimistic).to(torch.float32) + 1


@torch.no_grad()
def ranking_metrics(rank):
    """reference train/evaluation.py:23-50 from the ranks: Hits@{10,50,100} and MRR."""
    res = torch.stack([(rank <= 10).float().mean(), (rank <= 50).float().mean(), (rank <= 100).float().mean(),
                       (1.0 / rank).mean()]).tolist()
    return {"Hits@10": res[0], "Hits@50": res[1], "Hits@100": res[2], "MRR": res[3]}


@torch.no_grad()
def evaluate_mrr(y_pred_pos, y_pred_neg):
    """reference train/evaluation.py:23-50: Hits@{10,50,100} and MRR of the ranking list."""
    return ranking_metrics(get_ranking_list(y_pred_pos, y_pred_neg))


@torch.no_grad()
def evaluate_full_ranking(model, score_func, source, positive, X, exclude=None, test_set=False, group=None,
                          batch_size=None, stream=None):
    """Filtered full-ranking Hits@{10,50,100} and MRR: every positive (source[q], positive[q]) ranked among ALL nodes
    but the source and its row of `exclude` (top_targets_sharded) instead of among sampled negatives."""
    return ranking_metrics(top_targets_sharded(model, score_func, source, X, 1, exclude=exclude, positive=positive,
                                               test_set=test_set, group=group, batch_size=batch_size,
                                               stream=stream).rank)


@torch.no_grad()
def sample_level_hits(y_pred_pos, y_pred_neg):
    """reference train/evaluation.py:53-72: per-sample Hits@{20,50,100} (device tensors)."""
    rank = get_ranking_list(y_pred_pos, y_pred_neg)
    return {"Hits@20": (rank <= 20).float(), "Hits@50": (rank <= 50).float(), "Hits@100": (rank <= 100).float()}


@torch.no_grad()
def evaluate_hits(evaluator, pos_pred, neg_pred, k_list):
    """reference train/evaluation.py:7-20 with OGB's Hits@K (ogb/linkproppred/evaluate.py `_eval_hits`: a positive is a
    hit if it scores above the K-th highest negative; 1.0 when there are fewer than K negatives) computed on the
    device for every K at once.  `evaluator` is accepted for signature compatibility and not called."""
    pos, neg = pos_pred.reshape(-1), neg_pred.reshape(-1)
    ks = [int(k) for k in k_list]
    top = torch.topk(neg, min(max(ks), neg.numel()))[0] if neg.numel() > 0 else neg
    vals = []
    for k in ks:
        if neg.numel() < k:
            vals.append(torch.ones((), device=pos.device))
        else:
            vals.append((pos > top[k - 1]).float().sum() / max(1, pos.numel()))
    vals = torch.stack(vals).tolist()
    return {f"Hits@{k}": v for k, v in zip(ks, vals)}


@torch.no_grad()
def evaluate_auc(val_pred, val_true):
    """reference train/evaluation.py:93-105 (sklearn roc_auc_score / average_precision_score, rounded to 4 places) on
    the device: AUC from the rank-sum statistic with average ranks for ties, AP as the step-wise sum over the
    distinct thresholds."""
    pred = val_pred.reshape(-1).to(torch.float64)
    true = val_true.reshape(-1).to(pred.device) > 0
    n_pos, n_neg = int(true.sum()), int((~true).sum())
    vals, inv, cnt = torch.unique(pred, return_inverse=True, return_counts=True)       # ascending distinct scores
    end = torch.cumsum(cnt, 0).to(torch.float64)
    avg_rank = end - (cnt.to(torch.float64) - 1) / 2                                   # average 1-based rank of a tie group
    auc = (avg_rank[inv][true].sum() - n_pos * (n_pos + 1) / 2) / max(1, n_pos * n_neg)
    # precision / recall at every distinct threshold, from the highest score down
    pos_per = torch.zeros_like(end).index_add_(0, inv, true.to(torch.float64)).flip(0)
    tp = torch.cumsum(pos_per, 0)
    seen = torch.cumsum(cnt.flip(0), 0).to(torch.float64)
    ap = (pos_per / max(1, n_pos) * (tp / seen)).sum()
    auc, ap = torch.stack([auc, ap]).tolist()
    return {"AUC": round(auc, 4), "AP": round(ap, 4)}


def get_metric_score(evaluator_hit, evaluator_mrr, pos_train_pred, pos_val_pred, neg_val_pred, pos_test_pred, neg_test_pred,
                     k_list=[100]):
    """reference train/evaluation.py:108-130 (the MRR variant ranks every positive against the whole negative list)."""
    result = {}
    hit_train = evaluate_hits(evaluator_hit, pos_train_pred, neg_val_pred, k_list)
    hit_val = evaluate_hits(evaluator_hit, pos_val_pred, neg_val_pred, k_list)
    hit_test = evaluate_hits(evaluator_hit, pos_test_pred, neg_test_pred, k_list)
    for K in k_list:
        result[f"Hits@{K}"] = (hit_train[f"Hits@{K}"], hit_val[f"Hits@{K}"], hit_test[f"Hits@{K}"])
    if evaluator_mrr is not None:
        result["MRR"] = (evaluate_mrr(pos_train_pred, neg_val_pred.reshape(1, -1))["MRR"],
                         evaluate_mrr(pos_val_pred, neg_val_pred.reshape(1, -1))["MRR"],
                         evaluate_mrr(pos_test_pred, neg_test_pred.reshape(1, -1))["MRR"])
    return result


def get_metric_score_citation2(evaluator_mrr, pos_train_pred, pos_val_pred, neg_val_pred, pos_test_pred, neg_test_pred):
    """reference train/evaluation.py:133-148."""
    return {"MRR": (evaluate_mrr(pos_train_pred, neg_val_pred)["MRR"], evaluate_mrr(pos_val_pred, neg_val_pred)["MRR"],
                    evaluate_mrr(pos_test_pred, neg_test_pred)["MRR"])}


# ------------------------------------------------------------------------------------------------------------
# Eval drivers (reference train/testing.py), same names and arguments; the batch loops are LinkScoreStreams and the
# predictions are device tensors (the reference's per-batch .cpu() is what caps its throughput).
# ------------------------------------------------------------------------------------------------------------
@torch.no_grad()
def test_edge_citation2(model, score_func, input_data, h, batch_size, mrr_mode=False, negative_data=None, test=False,
                        stream=None):
    """reference train/testing.py:14-47 with the batch loop pipelined (LinkScoreStream) and the predictions kept
    on the device.  input_data [P, 2] positive edges; mrr_mode: negative_data [P, K] negative targets of each
    positive's source, result [P, K]; else result [P].  The negatives are scored as query groups (score_grouped:
    each positive's source with its K targets), never as a [2, P*K] pair tensor."""
    dev = h.device
    st = stream if stream is not None else LinkScoreStream(model, score_func, h, batch_size, test_set=test)
    if mrr_mode:
        targets = negative_data.to(dev)
        if targets.dtype not in (torch.int32, torch.int64):
            targets = targets.long()
        return st.score_grouped(input_data[:, 0].to(dev, targets.dtype), targets)
    return st.score(input_data.t().to(dev).contiguous())


@torch.no_grad()
def test_citation2(model, score_func, data, evaluator_hit, evaluator_mrr, batch_size):
    """reference train/testing.py:50-74 (citation2: propagate once; the train predictions are overwritten by the
    validation ones there, :70 — kept, parity first)."""
    model.eval()
    score_func.eval()
    h = model.propagate()
    neg_valid_pred = test_edge_citation2(model, score_func, data["valid_pos"], h, batch_size, mrr_mode=True, negative_data=data["valid_neg"])
    pos_valid_pred = test_edge_citation2(model, score_func, data["valid_pos"], h, batch_size)
    pos_test_pred = test_edge_citation2(model, score_func, data["test_pos"], h, batch_size, test=True)
    neg_test_pred = test_edge_citation2(model, score_func, data["test_pos"], h, batch_size, mrr_mode=True, negative_data=data["test_neg"], test=True)
    test_edge_citation2(model, score_func, data["train_pos_val"], h, batch_size)
    pos_valid_pred = pos_valid_pred.view(-1)
    pos_test_pred = pos_test_pred.view(-1)
    pos_train_pred = pos_valid_pred.view(-1)
    return get_metric_score_citation2(evaluator_mrr, pos_train_pred, pos_valid_pred, neg_valid_pred, pos_test_pred, neg_test_pred)


@torch.no_grad()
def test_edge(model, score_func, input_data, batch_size, test_set=False, dump_att=False):
    """reference train/testing.py:77-92.  The reference calls model(edge, test_set) per batch, i.e. re-runs the GCN on
    the train (or, for test_set, the full) graph every time (:87 -> link_transformer.py:100); the embeddings do not
    depend on the batch, so they are computed once here.  input_data [P, 2]; returns [P] scores on the device."""
    h = model.propagate(test_set=test_set)
    links = input_data.t().to(h.device).contiguous()
    return LinkScoreStream(model, score_func, h, batch_size, test_set=test_set).score(links)


@torch.no_grad()
def test_heart_negatives(negative_data, model, score_func, batch_size=32768, test_set=False):
    """reference train/testing.py:95-121 (HeaRT): negative_data [P, K, 2] -> scores [P, K].  As in the reference the
    embeddings come from the TRAIN graph (h = model.propagate(), :105) also when test_set selects the full tables for
    the pairwise part."""
    num_negative = negative_data.size(1)
    h = model.propagate()
    links = torch.permute(negative_data, (2, 0, 1)).reshape(2, -1).to(h.device).contiguous()
    return LinkScoreStream(model, score_func, h, batch_size, test_set=test_set).score(links).view(-1, num_negative)


@torch.no_grad()
def test(model, score_func, data, evaluator_hit, evaluator_mrr, batch_size, k_list=[100], heart=False, dump_att=False,
         dump_test=False, metric="Hits@100"):
    """reference train/testing.py:124-173."""
    model.eval()
    score_func.eval()
    pos_train_pred = test_edge(model, score_func, data["train_pos_val"], batch_size)
    pos_valid_pred = test_edge(model, score_func, data["valid_pos"], batch_size)
    pos_test_pred = test_edge(model, score_func, data["test_pos"], batch_size, test_set=True, dump_att=dump_att)
    if heart:
        neg_valid_pred = test_heart_negatives(data["valid_neg"], model, score_func, batch_size=batch_size)
        neg_test_pred = test_heart_negatives(data["test_neg"], model, score_func, batch_size=batch_size, test_set=True)
        result = get_metric_score_citation2(evaluator_mrr, pos_train_pred.view(-1), pos_valid_pred.view(-1), neg_valid_pred,
                                            pos_test_pred.view(-1), neg_test_pred)
    else:
        neg_valid_pred = test_edge(model, score_func, data["valid_neg"], batch_size)
        neg_test_pred = test_edge(model, score_func, data["test_neg"], batch_size, test_set=True, dump_att=dump_att)
        result = get_metric_score(evaluator_hit, evaluator_mrr, pos_train_pred, torch.flatten(pos_valid_pred),
                                  torch.flatten(neg_valid_pred), pos_test_pred, neg_test_pred, k_list)
    if dump_test:
        return result, sample_level_hits(pos_test_pred, neg_test_pred)[metric]
    return result
