"""Tensor-level wrappers over the C-ABI (one function per entry point).

All tensors must live on the CUDA device; outputs are allocated with torch (device memory
plumbing) and every launch goes to torch's current stream.
"""
from __future__ import annotations

import os
from dataclasses import dataclass
from typing import Optional

import torch

from . import _lib
from ._lib import EPI_NONE, EPI_RELU, EPI_SIGMOID, MODE, call, ptr, require_cuda, stream
from .graph import CSR

TYPE_NAMES = ("cn", "1hop", "non1hop")


def _rowmajor(x: torch.Tensor) -> torch.Tensor:
    """fp32 2-D tensor with unit stride in the last dimension (row stride arbitrary)."""
    if x.dtype != torch.float32:
        x = x.float()
    if x.dim() != 2:
        raise ValueError("expected a 2-D tensor")
    if x.stride(1) != 1 or x.stride(0) < x.shape[1]:
        x = x.contiguous()
    return x


def gemm(A, W, bias=None, bias_scale=1.0, out=None, epilogue=EPI_NONE):
    """out[M,N] = epi(A[M,K] @ W[N,K]^T + bias_scale * bias)."""
    require_cuda(A, W, bias, out)
    A, W = _rowmajor(A), _rowmajor(W)
    M, K = A.shape
    N = W.shape[0]
    if W.shape[1] != K:
        raise ValueError(f"gemm: A is [{M},{K}] but W is {list(W.shape)}")
    if out is None:
        out = torch.empty((M, N), dtype=torch.float32, device=A.device)
    elif out.shape != (M, N) or out.stride(1) != 1 or out.dtype != torch.float32:
        raise ValueError("gemm: bad `out`")
    if bias is not None:
        bias = bias.float().contiguous()
    call("lpf_gemm", ptr(A), A.stride(0), ptr(W), W.stride(0), ptr(bias), float(bias_scale), ptr(out),
         out.stride(0) if M > 0 else N, M, N, K, epilogue, stream(), meta=(M, N, K))
    return out


_PACKED = {}          # (data_ptr, version, shape, stride) -> (packed image, weight kept alive)
USE_PACKED_ROWS = os.environ.get("LPF_PACKED_ROWS", "1") != "0"   # one-pass selection over the packed link rows
GEMM_BACKEND = os.environ.get("LPF_GEMM_BACKEND", "tc")   # "tc": tcgen05 3xTF32 kernel (lpf_gemm_tc);  "simt": fp32 FFMA kernel (lpf_gemm)


def pack_weight(W):
    """Pre-split (hi/lo tf32) pre-swizzled image of an nn.Linear weight [N,K] for lpf_gemm_tc; cached per
    (storage, version) so it is built once per weight."""
    key = (W.data_ptr(), W._version, tuple(W.shape), W.stride(0), W.device.index)
    hit = _PACKED.get(key)
    if hit is not None:
        return hit[0]
    require_cuda(W)
    Wc = _rowmajor(W.detach())
    N, K = Wc.shape
    nbytes = _lib.load().lpf_pack_weight_bytes(N, K)
    packed = torch.empty(nbytes // 4, dtype=torch.float32, device=W.device)
    call("lpf_pack_weight", ptr(Wc), Wc.stride(0), N, K, ptr(packed), stream())
    if len(_PACKED) > 512:
        _PACKED.clear()
    _PACKED[key] = (packed, W)
    return packed


HEADS_F16 = os.environ.get("LPF_HEADS", "f16") != "tf32"   # d = 64 heads: fp16-split operands (lpf_link_heads_f16) or 3xTF32


def pow2_scale(bound, target_exp=15):
    """Largest power of two s with bound * s < 2^target_exp (1.0 for a zero bound)."""
    import math
    if not (bound > 0.0) or not math.isfinite(bound):
        return 1.0
    return 2.0 ** (target_exp - 1 - math.floor(math.log2(bound)))


def pack_weight_f16(W):
    """(image, scale): fp16 hi / lo images of an nn.Linear weight [N, K] in the swizzled K-major layout of
    tcgen05.mma.kind::f16 (lpf_pack_weight_f16), scaled by the power of two that puts max|W| into [2^14, 2^15)."""
    require_cuda(W)
    Wc = _rowmajor(W.detach())
    N, K = Wc.shape
    scale = pow2_scale(float(Wc.abs().max()))
    nbytes = _lib.load().lpf_pack_weight_f16_bytes(N, K)
    packed = torch.empty(nbytes // 4, dtype=torch.float32, device=W.device)
    call("lpf_pack_weight_f16", ptr(Wc), Wc.stride(0), N, K, float(scale), ptr(packed), stream())
    return packed, scale


def heads_call(links, bs, idx, n, X, c, zb, ld_zb, prob, logits, n_dev, sched, st):
    """One launch of the fused heads with the operand set `c` (model._head_consts): the fp16-split kernel when the
    consts carry its images (d = 64), the 3xTF32 kernel otherwise.  idx / zb / n_dev / sched: raw pointers or None."""
    d = X.shape[1]
    bf = X.dtype == torch.bfloat16
    if "w1h" in c and X.data_ptr() % 16 == 0 and (X.stride(0) * X.element_size()) % 16 == 0:
        call("lpf_link_heads_f16", ptr(links), bs, idx, n, ptr(X), int(bf), X.stride(0), X.shape[0], d, ptr(c["w1h"]), c["inv_sw1"], ptr(c["b1"]),
             ptr(c["ln_w_s"]), ptr(c["ln_b_s"]), ptr(c["w23h"]), c["inv_s3"], ptr(c["c3"]) if zb is None else None, zb, ld_zb,
             ptr(c["ws2"]), ptr(c["bs2"]), ptr(prob), int(logits), n_dev, st, meta=(n,),
             label=None if zb is None else "non-empty links (per-row offsets)")
    else:
        if bf:
            raise _lib.LpfError("bf16 node tables need the fp16-split heads (d = 64, 16-byte aligned rows)")
        call("lpf_link_heads_tc", ptr(links), bs, idx, n, ptr(X), X.stride(0), d, ptr(c["w1p"]), ptr(c["b1"]),
             ptr(c["ln_w"]), ptr(c["ln_b"]), ptr(c["w23p"]), ptr(c["c3"]) if zb is None else None, zb, ld_zb,
             ptr(c["ws2"]), ptr(c["bs2"]), ptr(prob), int(logits), n_dev, sched, st, meta=(n,),
             label=None if zb is None else "non-empty links (per-row offsets)")


def linear(A, W, bias=None, bias_scale=1.0, out=None, epilogue=EPI_NONE):
    """out[M,N] = epi(A @ W^T + bias_scale*bias) on the tensor cores (rows of W in chunks of <= 256)."""
    if GEMM_BACKEND != "tc":
        return gemm(A, W, bias, bias_scale, out, epilogue)
    require_cuda(A, W, bias, out)
    A = _rowmajor(A)
    M, K = A.shape
    N = W.shape[0]
    if W.shape[1] != K:
        raise ValueError(f"linear: A is [{M},{K}] but W is {list(W.shape)}")
    if out is None:
        out = torch.empty((M, N), dtype=torch.float32, device=A.device)
    elif out.shape != (M, N) or out.stride(1) != 1 or out.dtype != torch.float32:
        raise ValueError("linear: bad `out`")
    if bias is not None:
        bias = bias.detach().float().contiguous()
    for n0 in range(0, N, 256):
        n1 = min(N, n0 + 256)
        Wc = W if (n0 == 0 and n1 == N) else W[n0:n1]
        o = out if (n0 == 0 and n1 == N) else out[:, n0:n1]
        b = None if bias is None else (bias if (n0 == 0 and n1 == N) else bias[n0:n1])
        call("lpf_gemm_tc", ptr(A), A.stride(0), ptr(pack_weight(Wc)), ptr(b), float(bias_scale), ptr(o),
             o.stride(0) if M > 0 else N, M, n1 - n0, K, epilogue, None, stream(), meta=(M, n1 - n0, K))
    return out


def layernorm_act(x, weight, bias, relu=False, residual=None, out=None, n=None, dropout=None, row0=0):
    """out = residual + act(LayerNorm(x[:, :n])) row-wise; weight=None skips the norm.  dropout = (p, seed, site):
    out = residual + drop(act(LayerNorm(x))) with mask rows row0 + r (lpf_layernorm_act_dropout)."""
    require_cuda(x, weight, bias, residual, out)
    x = _rowmajor(x)
    rows = x.shape[0]
    n = x.shape[1] if n is None else n
    if out is None:
        out = torch.empty((rows, n), dtype=torch.float32, device=x.device)
    if residual is not None:
        residual = _rowmajor(residual)
    if dropout is not None:
        p, seed, site = dropout
        check_p(p)
        require_cuda(seed)
        call("lpf_layernorm_act_dropout", ptr(x), x.stride(0), ptr(weight), ptr(bias), int(relu), int(row0), ptr(seed),
             int(site), float(p), ptr(residual), residual.stride(0) if residual is not None else 0, ptr(out),
             out.stride(0), rows, n, stream())
        return out
    call("lpf_layernorm_act", ptr(x), x.stride(0), ptr(weight), ptr(bias), ptr(residual),
         residual.stride(0) if residual is not None else 0, ptr(out), out.stride(0), rows, n, int(relu), None, stream())
    return out


def gather_links(links, X, want_sum=True, want_prod=True, out_sum=None, out_prod=None, idx=None):
    """xsum = X[a]+X[b], xprod = X[a]*X[b] for every link, or for the batch positions listed in idx."""
    require_cuda(links, X, idx)
    X = _rowmajor(X)
    bs, d = links.shape[1], X.shape[1]
    n = bs if idx is None else idx.numel()
    if want_sum and out_sum is None:
        out_sum = torch.empty((n, d), dtype=torch.float32, device=X.device)
    if want_prod and out_prod is None:
        out_prod = torch.empty((n, d), dtype=torch.float32, device=X.device)
    call("lpf_gather_links", ptr(links), bs, ptr(idx), n, ptr(X), X.stride(0), d, ptr(out_sum),
         out_sum.stride(0) if out_sum is not None else 0, ptr(out_prod),
         out_prod.stride(0) if out_prod is not None else 0, None, int(X.dtype == torch.bfloat16), stream())
    return out_sum, out_prod


def scatter_rows(src, idx, dst, fill_row=None):
    """dst[:, :] = fill_row (if given), then dst[idx[j], :] = src[j, :]."""
    require_cuda(src, idx, dst, fill_row)
    n = 0 if idx is None or src is None else idx.numel()
    d = dst.shape[1]
    call("lpf_scatter_rows", ptr(src), src.stride(0) if n > 0 else d, ptr(idx), n, ptr(dst), dst.stride(0), dst.shape[0], d,
         ptr(fill_row), stream())
    return dst


@dataclass
class Selection:
    """Selected (link, node) pairs of one batch, type-major (CN | 1-hop | >1-hop), each type
    sorted by (link, node): the concatenation order of reference link_transformer.py:161."""
    mode: str
    bs: int
    ptr: torch.Tensor            # int64 [3*bs+1]
    node: torch.Tensor           # int32 [S]
    src_ppr: torch.Tensor        # fp32 [S]
    tgt_ppr: torch.Tensor        # fp32 [S]
    link: Optional[torch.Tensor]  # int32 [S] or None
    bounds: tuple                # (0, S_cn, S_cn+S_1hop, S) python ints
    nz: Optional[torch.Tensor] = None   # int32 [M']: batch positions of the links with a non-empty set (any order)

    @property
    def total(self) -> int:
        return self.bounds[3]

    def type_range(self, t: int):
        return self.bounds[t], self.bounds[t + 1]

    def counts(self) -> torch.Tensor:
        """int64 [3, bs] set sizes."""
        p = self.ptr
        return (p[1:] - p[:-1]).view(3, self.bs)


def merge_selections(near: Selection, far: Selection) -> Selection:
    """CN and 1-hop sets of `near` with the >1-hop sets of `far` (two selections of the same batch over different
    adjacency tables: a caller-supplied one decides CN / 1-hop, the stored one the >1-hop set — reference
    models/link_transformer.py:226-254 vs :443-447).  Slow path (torch ops, one host sync)."""
    bs, dev = near.bs, near.node.device
    cn, hop = near.counts()[0], near.counts()[1]
    far_cnt = far.counts()[2]
    counts = torch.cat((cn, hop, far_cnt))
    p = torch.zeros(3 * bs + 1, dtype=torch.int64, device=dev)
    p[1:] = torch.cumsum(counts, 0)
    n0, n1 = near.bounds[1], near.bounds[2]
    f0, f1 = far.bounds[2], far.bounds[3]
    cat = lambda a, b: torch.cat((a[:n1], b[f0:f1]))    # noqa: E731
    link = None if near.link is None or far.link is None else cat(near.link, far.link)
    nz = torch.nonzero((cn + hop + far_cnt) > 0).reshape(-1).to(torch.int32)
    return Selection("all", bs, p, cat(near.node, far.node), cat(near.src_ppr, far.src_ppr), cat(near.tgt_ppr, far.tgt_ppr),
                     link, (0, n0, n1, n1 + (f1 - f0)), nz)


def drop_packed_weights():
    """Forgets every cached tensor-core weight image (LinkTransformer.invalidate_weights)."""
    _PACKED.clear()
    _PACKED_T.clear()


def links_tensor(batch, device) -> torch.Tensor:
    """int64 [2,BS] contiguous on `device` (reference forward() moves the batch, :98)."""
    b = torch.as_tensor(batch)
    if b.dim() != 2 or b.shape[0] != 2:
        raise ValueError("batch must be a [2, BS] tensor of (source, target) node ids")
    return b.to(device=device, dtype=torch.int64).contiguous()


def query_groups(source, targets):
    """(source [Q], targets [Q, K]) of the grouped form, both int32 or both int64 and on the same device, contiguous.
    The flat link index q * K + j is link (source[q], targets[q, j]): the order of the reference's source.repeat(K)."""
    s, t = torch.as_tensor(source), torch.as_tensor(targets)
    if s.dim() != 1 or t.dim() != 2 or t.shape[0] != s.shape[0]:
        raise ValueError("query groups must be source [Q] and targets [Q, K] (one source and K targets per query); got "
                         f"{list(s.shape)} and {list(t.shape)}")
    if s.dtype != t.dtype or s.dtype not in (torch.int32, torch.int64):
        raise ValueError(f"source and targets must both be int32 or both int64; got {s.dtype} and {t.dtype}")
    if s.device != t.device:
        raise ValueError(f"source and targets must be on the same device; got {s.device} and {t.device}")
    return s.contiguous(), t.contiguous()


def expand_query_links(source, targets, K, j0, n, num_nodes, links, bad):
    """links[:, :n] = the flat range of n links of the grouped form that starts at position j0 of its first query
    (lpf_expand_query_links).  source: ids from the first query the range touches on; targets: ids from the range's
    first target (both 1-D, contiguous, int32 or int64 alike); links: int64 [2, >= n] with unit stride in a row.  Ids
    outside [0, num_nodes) come out as 0 and set bad (int64 [1]); the caller resets it."""
    require_cuda(source, targets, links, bad)
    if source.dtype != targets.dtype or source.dtype not in (torch.int32, torch.int64):
        raise ValueError(f"source and targets must both be int32 or both int64; got {source.dtype} and {targets.dtype}")
    if not (source.is_contiguous() and targets.is_contiguous()):
        raise ValueError("source and targets must be contiguous")
    if links.dtype != torch.int64 or links.dim() != 2 or links.shape[0] != 2 or links.stride(1) != 1 or links.shape[1] < n:
        raise ValueError(f"links must be int64 [2, >= {n}] with unit stride in a row")
    if bad.dtype != torch.int64 or bad.numel() < 1:
        raise ValueError("bad must be an int64 device word")
    if n > 0 and K >= 1 and (targets.numel() < n or source.numel() < (j0 + n + K - 1) // K):
        raise ValueError(f"the range of {n} links at position {j0} needs {(j0 + n + K - 1) // K} sources and {n} targets; "
                         f"got {source.numel()} and {targets.numel()}")
    call("lpf_expand_query_links", ptr(source), ptr(targets), source.element_size(), int(K), int(j0), int(n),
         int(num_nodes), ptr(links), links.stride(0), ptr(bad), stream(), meta=(n,))
    return links


def _ids(name, t):
    if t.dtype not in (torch.int32, torch.int64) or t.dim() != 1 or not t.is_contiguous():
        raise ValueError(f"{name} must be a contiguous 1-D int32 or int64 tensor; got {t.dtype} {list(t.shape)}")


def expand_source_sweep(source, n_targets, j0, n, num_nodes, links, bad):
    """links[:, :n] = the flat range of n links of the source sweep (link q * n_targets + j is (source[q], j)) that
    starts at position j0 of its first query (lpf_expand_source_sweep).  source: ids from the first query the range
    touches on (1-D, contiguous, int32 or int64); links: int64 [2, >= n] with unit stride in a row.  A source outside
    [0, num_nodes) comes out as 0 and sets bad (int64 [1]); the caller resets it."""
    _ids("source", source)
    if links.dtype != torch.int64 or links.dim() != 2 or links.shape[0] != 2 or links.stride(1) != 1 or links.shape[1] < n:
        raise ValueError(f"links must be int64 [2, >= {n}] with unit stride in a row")
    if bad.dtype != torch.int64 or bad.numel() < 1:
        raise ValueError("bad must be an int64 device word")
    if n > 0 and n_targets >= 1 and source.numel() < (j0 + n + n_targets - 1) // n_targets:
        raise ValueError(f"the range of {n} links at position {j0} needs {(j0 + n + n_targets - 1) // n_targets} "
                         f"sources; got {source.numel()}")
    require_cuda(source, links, bad)
    call("lpf_expand_source_sweep", ptr(source), source.element_size(), int(n_targets), int(j0), int(n),
         int(num_nodes), ptr(links), links.stride(0), ptr(bad), stream(), meta=(n,))
    return links


def topk_fold_workspace(bs, k, n_targets, device):
    """A workspace for lpf_topk_fold over ranges of up to bs scores."""
    nbytes = _lib.load().lpf_topk_fold_workspace_bytes(int(bs), int(k), int(n_targets))
    if nbytes < 0:
        raise ValueError(f"bad top-k workspace arguments (bs {bs}, k {k}, n_targets {n_targets}; 1 <= k <= 1024)")
    return torch.empty(max(1, nbytes), dtype=torch.uint8, device=device)


def topk_fold(prob, lo, source, n_targets, k, top_key, top_id, workspace, exclude=None, positive=None,
              pos_score=None, cnt_ge=None, cnt_gt=None, skip=None):
    """Folds prob [n] — the scores of the sweep positions [lo, lo + n) — into the per-query state (lpf_topk_fold):
    top_key fp32 / top_id int32 [Q, k] (the k best candidates, score descending then id ascending; (-inf, -1) while
    unfilled) and, with positive [Q] / pos_score fp32 [Q], cnt_ge / cnt_gt int64 [Q] (candidates with score >= / > the
    positive's).  Candidates: every target in [0, n_targets) but the source and its row of `exclude` (a CSR or None);
    the counters also leave out the positive.  skip: an int64 device word; non-zero at launch time = fold nothing."""
    _ids("source", source)
    Q = source.numel()
    if prob.dtype != torch.float32 or prob.dim() != 1 or not prob.is_contiguous():
        raise ValueError("prob must be a contiguous fp32 [n] tensor")
    if not 1 <= int(k) <= 1024:
        raise ValueError(f"k must be in [1, 1024]; got {k}")
    if top_key.dtype != torch.float32 or top_id.dtype != torch.int32 or tuple(top_key.shape) != (Q, k) or \
            tuple(top_id.shape) != (Q, k) or not (top_key.is_contiguous() and top_id.is_contiguous()):
        raise ValueError(f"top_key / top_id must be contiguous fp32 / int32 [{Q}, {k}]")
    given = [t is not None for t in (positive, pos_score, cnt_ge, cnt_gt)]
    if any(given) and not all(given):
        raise ValueError("positive, pos_score, cnt_ge and cnt_gt go together")
    if positive is not None:
        _ids("positive", positive)
        if positive.dtype != source.dtype or positive.numel() != Q:
            raise ValueError(f"positive must be [{Q}] of the source's dtype ({source.dtype})")
        if pos_score.dtype != torch.float32 or pos_score.numel() != Q or not pos_score.is_contiguous():
            raise ValueError(f"pos_score must be a contiguous fp32 [{Q}] tensor")
        for c in (cnt_ge, cnt_gt):
            if c.dtype != torch.int64 or c.numel() != Q or not c.is_contiguous():
                raise ValueError(f"cnt_ge / cnt_gt must be contiguous int64 [{Q}] tensors")
    if skip is not None and (skip.dtype != torch.int64 or skip.numel() < 1):
        raise ValueError("skip must be an int64 device word")
    require_cuda(prob, source, top_key, top_id, workspace, positive, pos_score, cnt_ge, cnt_gt, skip)
    if exclude is not None:
        require_cuda(exclude.rowptr, exclude.col)
        if exclude.nnz == 0:          # (no row to look up; an empty col may have no storage)
            exclude = None
    n = prob.numel()
    call("lpf_topk_fold", ptr(prob), int(lo), n, ptr(source), ptr(positive), source.element_size(), Q, int(n_targets),
         None if exclude is None else ptr(exclude.rowptr), None if exclude is None else ptr(exclude.col),
         0 if exclude is None else exclude.n, ptr(pos_score), int(k), ptr(top_key), ptr(top_id), ptr(cnt_ge),
         ptr(cnt_gt), ptr(skip), ptr(workspace), workspace.numel(), stream(), meta=(n,))


def pick_select_algo(adj: CSR, ppr: CSR, th_1hop, th_non1hop, mode: str) -> int:
    """Intersection-driven kernel when its preconditions hold (thresholds gating PPR-derived sets > 0 and
    all PPR values in (0,1], checked once per table), group width by mean row length; else the generic one."""
    ok = mode == "cn" or (th_1hop > 0 and (mode != "all" or th_non1hop > 0))
    if not ok:
        return _lib.ALGO_GENERIC
    if ppr.unit_range is None:
        ppr.unit_range = bool(ppr.val.numel() == 0 or (float(ppr.val.min()) > 0.0 and float(ppr.val.max()) <= 1.0))
    if not ppr.unit_range:
        return _lib.ALGO_GENERIC
    # rows walked per link: adjacency rows, and the PPR rows when the mode has PPR-derived sets — a group defers a link
    # whose shorter row exceeds 16 elements per lane to the CTA-wide kernel, so long PPR rows (ogbl-collab shape: ~325
    # entries) on a sparse graph want full warps too (measured there: every link deferred with groups of 8, 1.5 ms of
    # CTA-wide walks per 32,565-link batch)
    mean_row = adj.nnz / max(1, adj.n)
    if mode != "cn":
        mean_row = max(mean_row, ppr.nnz / max(1, ppr.n))
    return _lib.ALGO_INTERSECT32 if mean_row >= 96 else _lib.ALGO_INTERSECT8


def select(links, adj: CSR, ppr: CSR, th_cn, th_1hop, th_non1hop, mode: str, want_link=False, algo=None) -> Selection:
    """K1: count -> scan -> fill.  One host sync (reading the three totals) sizes the outputs."""
    require_cuda(links, adj.rowptr, ppr.rowptr)
    dev = links.device
    bs = links.shape[1]
    m = MODE[mode]
    st = stream()
    counts = torch.empty(3 * bs, dtype=torch.int32, device=dev)
    args = (ptr(links), bs, ptr(adj.rowptr), ptr(adj.col), ptr(ppr.rowptr), ptr(ppr.col), ptr(ppr.val),
            float(th_cn), float(th_1hop), float(th_non1hop), m,
            pick_select_algo(adj, ppr, th_1hop, th_non1hop, mode) if algo is None else algo)
    ws = torch.empty(_lib.load().lpf_select_workspace_bytes(bs) // 4, dtype=torch.int32, device=dev)
    call("lpf_select_count", *args, ptr(counts), ptr(ws), st, meta=(bs,))
    p = torch.empty(3 * bs + 1, dtype=torch.int64, device=dev)
    scratch = torch.empty(max(1, _lib.load().lpf_scan_scratch_bytes(3 * bs) // 8), dtype=torch.int64, device=dev)
    call("lpf_scan_counts", ptr(counts), 3 * bs, ptr(p), ptr(scratch), st)
    nz = torch.empty(bs, dtype=torch.int32, device=dev)
    header = torch.empty(4, dtype=torch.int64, device=dev)
    call("lpf_select_compact", ptr(p), bs, ptr(nz), ptr(header), st)
    b = header.tolist()          # the one host sync of the batch: (S_cn, S_cn+S_1hop, S, #non-empty links)
    S = b[2]
    node = torch.empty(S, dtype=torch.int32, device=dev)
    pa = torch.empty(S, dtype=torch.float32, device=dev)
    pb = torch.empty(S, dtype=torch.float32, device=dev)
    link = torch.empty(S, dtype=torch.int32, device=dev) if want_link else None
    if S > 0:
        call("lpf_select_fill", *args, ptr(p), ptr(node), ptr(pa), ptr(pb), ptr(link), ptr(ws), st, meta=(bs, S))
    return Selection(mode, bs, p, node, pa, pb, link, (0, b[0], b[1], b[2]), nz[:b[3]])


class LinkRows:
    """Packed link rows of one (adjacency, PPR) table pair (lpf_pack_link_rows): `slab` = one 128-byte line per node
    (header + the first seven 16-byte chunks of its row) and `overflow` = the rest of the longer rows."""

    def __init__(self, adj: CSR, ppr: CSR):
        require_cuda(adj.rowptr, ppr.rowptr)
        lib = _lib.load()
        dev = adj.rowptr.device
        n = adj.n
        nbytes = lib.lpf_link_rows_bytes(n, adj.nnz, ppr.nnz)
        if nbytes < 0:
            raise _lib.LpfError("graph too large for the 32-bit unit index of the packed link rows")
        # (torch's caching allocator aligns to 512 bytes; the rows need 128)
        self.slab = torch.empty(max(lib.lpf_link_rows_slab_bytes(n) // 4, 32), dtype=torch.int32, device=dev)
        self.overflow = torch.empty(max(nbytes // 4, 32), dtype=torch.int32, device=dev)
        scratch = torch.empty(max(lib.lpf_link_rows_scratch_bytes(n) // 8 + 2, 2), dtype=torch.int64, device=dev)
        call("lpf_pack_link_rows", ptr(adj.rowptr), ptr(adj.col), ptr(ppr.rowptr), ptr(ppr.col), ptr(ppr.val), n,
             ptr(self.slab), ptr(self.overflow), ptr(scratch), stream())
        torch.cuda.current_stream().synchronize()     # scratch is released here
        self.adj, self.ppr = adj, ppr


def link_rows(adj: CSR, ppr: CSR) -> LinkRows:
    """The packed rows of (adj, ppr), built once per table pair and cached on the adjacency object."""
    cache = adj.__dict__.setdefault("_link_rows", {})
    key = id(ppr)
    lr = cache.get(key)
    if lr is None or lr.ppr is not ppr:
        lr = cache[key] = LinkRows(adj, ppr)
    return lr


def select_onepass(links, adj: CSR, ppr: CSR, th_cn, th_1hop, th_non1hop, mode: str, cap: int, algo=None):
    """K1, one launch sequence and no host round trip (lpf_select_onepass): pairs of type t land in rows
    [t*cap, t*cap + header[t]) of the pair arrays, per-link segments in (seg_start, counts).  Returns a dict of the
    raw device buffers; ScorePlan (plan.py) is the production caller, tests use this wrapper."""
    require_cuda(links, adj.rowptr, ppr.rowptr)
    dev = links.device
    bs = links.shape[1]
    algo = pick_select_algo(adj, ppr, th_1hop, th_non1hop, mode) if algo is None else algo
    out = {
        "counts": torch.empty(3 * bs, dtype=torch.int32, device=dev),
        "seg_start": torch.empty(3 * bs, dtype=torch.int32, device=dev),
        "nz": torch.empty(bs, dtype=torch.int32, device=dev),
        "header": torch.zeros(8, dtype=torch.int64, device=dev),
        "node": torch.empty(3 * cap, dtype=torch.int32, device=dev),
        "src_ppr": torch.empty(3 * cap, dtype=torch.float32, device=dev),
        "tgt_ppr": torch.empty(3 * cap, dtype=torch.float32, device=dev),
        "cap": cap,
    }
    ws = torch.empty(_lib.load().lpf_select_workspace_bytes(bs) // 4, dtype=torch.int32, device=dev)
    out["workspace"] = ws        # (word 0: deferred links; word bs + 4: candidates of the packed screening)
    if algo == _lib.ALGO_PACKED:
        lr = link_rows(adj, ppr)
        call("lpf_select_onepass_packed", ptr(links), bs, ptr(adj.rowptr), ptr(adj.col), ptr(ppr.rowptr), ptr(ppr.col),
             ptr(ppr.val), ptr(lr.slab), ptr(lr.overflow), float(th_cn), float(th_1hop), float(th_non1hop), MODE[mode], cap,
             ptr(out["counts"]), ptr(out["seg_start"]), ptr(out["nz"]), ptr(out["header"]), ptr(out["node"]),
             ptr(out["src_ppr"]), ptr(out["tgt_ppr"]), ptr(ws), stream(), meta=(bs,))
        return out
    call("lpf_select_onepass", ptr(links), bs, ptr(adj.rowptr), ptr(adj.col), ptr(ppr.rowptr), ptr(ppr.col), ptr(ppr.val),
         float(th_cn), float(th_1hop), float(th_non1hop), MODE[mode], algo, cap, ptr(out["counts"]),
         ptr(out["seg_start"]), ptr(out["nz"]), ptr(out["header"]), ptr(out["node"]), ptr(out["src_ppr"]),
         ptr(out["tgt_ppr"]), ptr(ws), stream(), meta=(bs,))
    return out


def rpe_hidden(sel: Selection, t: int, w1, b1, ln_w, ln_b, hsum):
    r0, r1 = sel.type_range(t)
    if r1 > r0:
        call("lpf_rpe_hidden", ptr(sel.src_ppr), ptr(sel.tgt_ppr), r0, r1 - r0, ptr(w1), ptr(b1), ptr(ln_w),
             ptr(ln_b), hsum.shape[1], ptr(hsum), hsum.stride(0), None, stream())


ATTEND_WS_BYTES = 4 << 20     # chunk records of the grid-wide split of giant links (lpf_attend_fused_ws)


def attend(sel: Selection, KV, R, Q, att, bias, ln_w, ln_b, heads, ch, write_counts, out, alpha_out=None, idx=None,
           r_map=None, r_const=None):
    """K4 over every link of the batch, or over the batch positions in idx (rows of Q / out follow idx).  With r_map
    (int32 [S]) R holds only the rows of the pairs the map points to; the others read r_const [3, H*C] by type."""
    require_cuda(KV, R, Q, out, idx, r_map, r_const)
    n = sel.bs if idx is None else idx.numel()
    # links with thousands of pairs are split over the grid through a workspace (lpf_attend_fused_ws)
    ws = torch.empty(ATTEND_WS_BYTES, dtype=torch.uint8, device=KV.device)
    call("lpf_attend_fused_ws", ptr(sel.ptr), sel.bs, ptr(idx), n, ptr(sel.node), ptr(KV), KV.stride(0),
         ptr(R) if sel.total > 0 else None, R.stride(0) if R is not None and R.dim() == 2 else heads * ch,
         ptr(Q), Q.stride(0), ptr(att), ptr(bias), ptr(ln_w), ptr(ln_b), heads, ch, MODE[sel.mode],
         int(write_counts), ptr(out), out.stride(0), ptr(alpha_out), None, None, None, 0,
         int(KV.dtype == torch.bfloat16), ptr(r_map), ptr(r_const), ptr(ws), ws.numel(), stream(),
         meta=(n, sel.total, heads * ch))
    return out


def link_heads(links, X, consts, prob, idx=None, zb=None, logits=False, sched=None):
    """Fused tensor-core heads (lpf_link_heads_f16 / lpf_link_heads_tc): prob[pos] for every link (constant pairwise half `c3`) or for the
    positions in idx with per-row zb.  `sched` (int32 [2], zeros): tiles handed out dynamically (see the header)."""
    require_cuda(links, X, prob, idx, zb, sched)
    X = _rowmajor(X)
    bs = links.shape[1]
    n = bs if idx is None else idx.numel()
    heads_call(links, bs, ptr(idx), n, X, consts, ptr(zb), zb.stride(0) if zb is not None else 0, prob, logits, None,
               ptr(sched), stream())
    return prob


def gcn_layer(adj: CSR, XW, bias, ln=None, relu=False, residual=None, ln2=None, out=None, row0=0, rows=None, local=False,
              dropout=None):
    """One GCN layer after its Linear, in one launch (lpf_gcn_layer): out = LN2(residual + act(LN(A_hat XW + bias)))
    for rows [row0, row0 + rows).  ln / ln2: (weight, bias) or None.  local=False: `out` and `residual` are [n, d]
    tables indexed by node id; local=True: they hold only the rows of the range (row 0 = node row0: the row-sharded
    multi-GPU layers).  dropout = (p, seed, site): out = LN2(residual + drop(act(LN(...)))), mask row = node id
    (lpf_gcn_layer_dropout).  Falls back to lpf_gcn_spmm + lpf_layernorm_act for widths / alignments the fused kernel
    does not take."""
    require_cuda(adj.rowptr, XW, bias, out, residual)
    if dropout is not None:
        check_p(dropout[0])
        require_cuda(dropout[1])
    XW = _rowmajor(XW)
    n, d = adj.n, XW.shape[1]
    rows = n - row0 if rows is None else rows
    if out is None:
        out = torch.empty((rows if local else n, d), dtype=torch.float32, device=XW.device)
    if residual is not None:
        residual = _rowmajor(residual)
    shift = row0 if local else 0          # the kernel indexes `out` / `residual` by node id
    a16 = lambda t: t is None or t.data_ptr() % 16 == 0     # noqa: E731
    fusable = d % 4 == 0 and d <= 512 and XW.stride(0) % 4 == 0 and out.stride(0) % 4 == 0 and a16(XW) and a16(out) and \
        a16(bias) and (residual is None or (a16(residual) and residual.stride(0) % 4 == 0)) and \
        all(a16(t) for pair in (ln, ln2) if pair is not None for t in pair)
    if fusable and dropout is not None:
        call("lpf_gcn_layer_dropout", ptr(adj.rowptr), ptr(adj.col), ptr(adj.val), row0, rows, ptr(XW), XW.stride(0),
             ptr(bias), d, ptr(ln[0]) if ln else None, ptr(ln[1]) if ln else None, int(relu), ptr(dropout[1]),
             int(dropout[2]), float(dropout[0]),
             (residual.data_ptr() - 4 * shift * residual.stride(0)) if residual is not None else None,
             residual.stride(0) if residual is not None else 0,
             ptr(ln2[0]) if ln2 else None, ptr(ln2[1]) if ln2 else None,
             out.data_ptr() - 4 * shift * out.stride(0), out.stride(0), stream(), meta=(rows, d, adj.nnz))
        return out
    if fusable:
        call("lpf_gcn_layer", ptr(adj.rowptr), ptr(adj.col), ptr(adj.val), row0, rows, ptr(XW), XW.stride(0), ptr(bias), d,
             ptr(ln[0]) if ln else None, ptr(ln[1]) if ln else None, int(relu),
             (residual.data_ptr() - 4 * shift * residual.stride(0)) if residual is not None else None,
             residual.stride(0) if residual is not None else 0,
             ptr(ln2[0]) if ln2 else None, ptr(ln2[1]) if ln2 else None,
             out.data_ptr() - 4 * shift * out.stride(0), out.stride(0), stream(), meta=(rows, d, adj.nnz))
        return out
    view = out if not local else None
    if local:       # unfused kernels index by node id: go through a full-height scratch table
        view = torch.empty((n, d), dtype=torch.float32, device=XW.device)
    gcn_spmm(adj, XW, bias, out=view, row0=row0, rows=rows)
    sh = view[row0:row0 + rows]
    dst = out if local else out[row0:row0 + rows]
    res = None if residual is None else (residual if local else residual[row0:row0 + rows])
    if ln is not None or relu or res is not None or dropout is not None:
        layernorm_act(sh, None if ln is None else ln[0], None if ln is None else ln[1], relu=relu, residual=res, out=dst,
                      dropout=dropout, row0=row0)
        sh = dst
    if ln2 is not None:
        layernorm_act(sh, ln2[0], ln2[1], relu=False, out=dst)
    elif sh is not dst:
        dst.copy_(sh)
    return out


def gcn_spmm(adj: CSR, XW, bias, out=None, row0=0, rows=None):
    require_cuda(adj.rowptr, XW, bias, out)
    XW = _rowmajor(XW)
    n, d = adj.n, XW.shape[1]
    rows = n - row0 if rows is None else rows
    if out is None:
        out = torch.empty((n, d), dtype=torch.float32, device=XW.device)
    call("lpf_gcn_spmm", ptr(adj.rowptr), ptr(adj.col), ptr(adj.val), row0, rows, ptr(XW), XW.stride(0), ptr(bias), d,
         ptr(out), out.stride(0), stream())
    return out


# ---------------------------------------------------------------------------------------------- backward (backward.cu)
def _workspace(nbytes, device):
    if nbytes < 0:
        raise ValueError("bad workspace arguments")
    return torch.empty(max(1, (nbytes + 15) // 16 * 4), dtype=torch.float32, device=device)


def layernorm_act_backward(x, weight, bias, dy, relu=False, dx=None, accumulate_dx=False, dweight=None, dbias=None,
                           accumulate_param=False, n=None):
    """Gradients of y = act(LN(x[:, :n])) (lpf_layernorm_act) from the saved pre-norm rows x: dx (written, or added with
    accumulate_dx) and, with weight, dweight / dbias (written, or added with accumulate_param).  Returns dx."""
    require_cuda(x, weight, bias, dy, dx, dweight, dbias)
    x, dy = _rowmajor(x), _rowmajor(dy)
    rows = x.shape[0]
    n = x.shape[1] if n is None else n
    if dx is None:
        dx = torch.empty((rows, n), dtype=torch.float32, device=x.device)
    ws = None
    if weight is not None:
        if dweight is None or dbias is None:
            raise ValueError("layernorm_act_backward: dweight and dbias are needed with weight")
        ws = _workspace(_lib.load().lpf_layernorm_act_backward_workspace_bytes(rows, n), x.device)
    call("lpf_layernorm_act_backward", ptr(x), x.stride(0), ptr(weight), ptr(bias), int(relu), ptr(dy), dy.stride(0),
         ptr(dx), dx.stride(0), int(accumulate_dx), ptr(dweight), ptr(dbias), int(accumulate_param), rows, n, ptr(ws),
         0 if ws is None else 4 * ws.numel(), stream(), meta=(rows, n),
         launches=0 if rows == 0 else (3 if weight is not None else 1))      # (with weight: + two reductions)
    return dx


def gemm_wgrad(A, dY, dW=None, db=None, accumulate=False):
    """dW (+)= dY^T A and db (+)= the column sums of dY (lpf_gemm_wgrad); A may be None when only db is wanted."""
    require_cuda(A, dY, dW, db)
    dY = _rowmajor(dY)
    M, N = dY.shape
    K = 1
    if dW is not None:
        A = _rowmajor(A)
        K = A.shape[1]
        if A.shape[0] != M or tuple(dW.shape) != (N, K) or dW.stride(1) != 1:
            raise ValueError(f"gemm_wgrad: A {list(A.shape)}, dY {list(dY.shape)}, dW {list(dW.shape)}")
    ws = _workspace(_lib.load().lpf_gemm_wgrad_workspace_bytes(M, N, K), dY.device)
    call("lpf_gemm_wgrad", ptr(A) if dW is not None else None, A.stride(0) if dW is not None else K, ptr(dY),
         dY.stride(0) if M > 0 else N, M, N, K, ptr(dW), dW.stride(0) if dW is not None else K, ptr(db), int(accumulate),
         ptr(ws), 4 * ws.numel(), stream(), meta=(M, N, K))


_PACKED_T = {}        # transposed weight images of linear_dgrad: (data_ptr, shape, stride, k0) -> (version, image, weight)


def linear_dgrad(dY, W, out=None, cache=True):
    """dX[M, K] = dY[M, N] @ W[N, K] on the tensor cores (lpf_gemm_tc on the packed transpose of W, in chunks of 256
    output columns).  cache=False for a W built for this call only: its image is not kept."""
    require_cuda(dY, W, out)
    dY = _rowmajor(dY)
    M, N = dY.shape
    K = W.shape[1]
    if W.shape[0] != N:
        raise ValueError(f"linear_dgrad: dY is [{M},{N}] but W is {list(W.shape)}")
    if out is None:
        out = torch.empty((M, K), dtype=torch.float32, device=dY.device)
    for k0 in range(0, K, 256):
        k1 = min(K, k0 + 256)
        key = (W.data_ptr(), tuple(W.shape), W.stride(0), W.device.index, k0)
        hit = _PACKED_T.get(key) if cache else None
        if hit is None or hit[0] != W._version or hit[2] is not W:     # (an optimizer step replaces the entry)
            Wt = W.detach()[:, k0:k1].t().contiguous()
            nbytes = _lib.load().lpf_pack_weight_bytes(k1 - k0, N)
            img = torch.empty(nbytes // 4, dtype=torch.float32, device=W.device)
            call("lpf_pack_weight", ptr(Wt), Wt.stride(0), k1 - k0, N, ptr(img), stream())
            hit = (W._version, img, W)
            if cache:
                if len(_PACKED_T) > 512:
                    _PACKED_T.clear()
                _PACKED_T[key] = hit
        o = out[:, k0:k1]
        call("lpf_gemm_tc", ptr(dY), dY.stride(0), ptr(hit[1]), None, 1.0, ptr(o), o.stride(0) if M > 0 else k1 - k0, M,
             k1 - k0, N, EPI_NONE, None, stream(), meta=(M, k1 - k0, N))
    return out


def act_backward(y, dy, act, out=None):
    """dx = dy [y > 0] (EPI_RELU) or dy y (1 - y) (EPI_SIGMOID) from the saved output y."""
    require_cuda(y, dy, out)
    y, dy = _rowmajor(y), _rowmajor(dy)
    rows, n = y.shape
    if out is None:
        out = torch.empty((rows, n), dtype=torch.float32, device=y.device)
    call("lpf_act_backward", ptr(y), y.stride(0), ptr(dy), dy.stride(0), ptr(out), out.stride(0), rows, n, act, stream())
    return out


def gather_links_backward(links, X, dX, dsum=None, dprod=None, idx=None):
    """dX[a] += dsum + dprod X[b], dX[b] += dsum + dprod X[a] for every link (or the positions in idx)."""
    require_cuda(links, X, dX, dsum, dprod, idx)
    X = _rowmajor(X)
    bs, d = links.shape[1], X.shape[1]
    n = bs if idx is None else idx.numel()
    dsum = None if dsum is None else _rowmajor(dsum)
    dprod = None if dprod is None else _rowmajor(dprod)
    call("lpf_gather_links_backward", ptr(links), bs, ptr(idx), n, ptr(X), X.stride(0), d, ptr(dsum),
         dsum.stride(0) if dsum is not None else 0, ptr(dprod), dprod.stride(0) if dprod is not None else 0, ptr(dX),
         dX.stride(0), stream(), meta=(n, d))
    return dX


def scatter_rows_backward(dG, idx, want_src=True):
    """(d src [n, d] or None, d fill_row [d]) of scatter_rows(src, idx, dst, fill_row)."""
    require_cuda(dG, idx)
    dG = _rowmajor(dG)
    rows, d = dG.shape
    n = 0 if idx is None else idx.numel()
    dsrc = torch.empty((n, d), dtype=torch.float32, device=dG.device) if want_src and n > 0 else None
    dfill = torch.empty(d, dtype=torch.float32, device=dG.device)
    ws = _workspace(_lib.load().lpf_scatter_rows_backward_workspace_bytes(rows, d), dG.device)
    call("lpf_scatter_rows_backward", ptr(dG), dG.stride(0), rows, d, ptr(idx), n, ptr(dsrc), d, ptr(dfill), ptr(ws),
         4 * ws.numel(), stream(), meta=(rows, d), launches=(1 if n > 0 else 0) + 2)   # gather + masked sum + reduction
    return dsrc, dfill


def rpe_hidden_backward(src_ppr, tgt_ppr, r0, r1, w1, b1, ln_w, ln_b, dh, grads, accumulate):
    """Adds (or writes) the gradients of one PPR encoder's first Linear + LayerNorm from dh = d hsum[r0:r1] (rows of dh
    in pair order).  grads: (dw1 [d, 2], db1, dln_w, dln_b)."""
    require_cuda(src_ppr, tgt_ppr, w1, dh, *grads)
    d = w1.shape[0]
    rows = r1 - r0
    dh = None if rows == 0 else _rowmajor(dh)
    ws = _workspace(_lib.load().lpf_rpe_hidden_backward_workspace_bytes(rows, d), w1.device)
    call("lpf_rpe_hidden_backward", ptr(src_ppr), ptr(tgt_ppr), r0, rows, ptr(w1), ptr(b1), ptr(ln_w), ptr(ln_b), d,
         ptr(dh), dh.stride(0) if rows > 0 else d, *[ptr(g) for g in grads], int(accumulate), ptr(ws), 4 * ws.numel(),
         stream(), meta=(rows, d))


def attend_backward(sel: Selection, KV, R, Q, att, bias, ln_w, ln_b, heads, ch, dY, dKV, idx=None, r_map=None,
                    r_const=None, dR=None, dR_const=None):
    """Backward of attend() (lpf_attend_backward): writes dR [rows of R, HC] (needed when R has rows), adds into
    dR_const [3, HC] (needed with r_map) and dKV [N, HC], and returns (dQ [n, HC], link_rows [n, 4 HC])."""
    require_cuda(KV, R, Q, dY, dKV, idx, r_map, r_const, dR, dR_const)
    n = sel.bs if idx is None else idx.numel()
    HC = heads * ch
    dev = KV.device
    dY = _rowmajor(dY)
    if R is None or R.shape[0] == 0:
        dR = None
    elif dR is None or dR.shape != R.shape or dR.stride(1) != 1:
        raise ValueError("attend_backward: dR must be a row-major table shaped like R")
    if (r_map is None) != (dR_const is None):
        raise ValueError("attend_backward: dR_const goes with r_map")
    dRc = dR_const
    dQ = torch.empty((n, HC), dtype=torch.float32, device=dev)
    rows = torch.empty((n, 4 * HC), dtype=torch.float32, device=dev)
    call("lpf_attend_backward", ptr(sel.ptr), sel.bs, ptr(idx), n, ptr(sel.node), ptr(KV), KV.stride(0),
         ptr(R) if dR is not None else None, R.stride(0) if dR is not None else HC, ptr(r_map), ptr(r_const), ptr(Q),
         Q.stride(0), ptr(att), ptr(bias), ptr(ln_w), ptr(ln_b), heads, ch, ptr(dY), dY.stride(0), ptr(dR),
         dR.stride(0) if dR is not None else HC, ptr(dRc), ptr(dQ), HC, ptr(dKV), dKV.stride(0), ptr(rows), stream(),
         meta=(n, sel.total, HC))
    return dQ, rows


# ------------------------------------------------------------------------------------------------ dropout (dropout.cu)
# site numbers of the dropout masks (include/lpformer_b200.h, "Dropout"): a mask is a function of (seed, site, row, col)
SITE_FEATURE, SITE_NODE, SITE_GCN, SITE_ATT, SITE_MLP = 1, 2, 16, 32, 48


def check_p(p):
    """F.dropout's argument check."""
    if not 0.0 <= float(p) <= 1.0:
        raise ValueError(f"dropout probability has to be between 0 and 1, but got {p}")


def draw_seed(device):
    """One 64-bit dropout seed from torch's CUDA generator of `device`, as an int64 [1] device tensor (no host sync):
    after torch.manual_seed(s) the same sequence of seeds, hence of masks, comes back."""
    return torch.randint(-2 ** 63, 2 ** 63 - 1, (1,), dtype=torch.int64, device=device)


def _seed_tensor(seed, device):
    if torch.is_tensor(seed):
        if seed.dtype != torch.int64 or seed.numel() < 1:
            raise ValueError("seed must be an int64 device tensor")
        require_cuda(seed)
        return seed
    return torch.tensor([int(seed) - (1 << 64) if int(seed) >= 1 << 63 else int(seed)], dtype=torch.int64, device=device)


def dropout(x, p, seed, site, row0=0, out=None):
    """out = x * mask / (1 - p) (lpf_dropout) over the rows of a 2-D fp32 tensor with unit column stride (any row stride);
    mask row = row0 + r.  out=x: in place.  seed: an int64 device tensor (draw_seed) or a Python int."""
    check_p(p)
    require_cuda(x, out)
    if x.dtype != torch.float32 or x.dim() != 2 or (x.shape[1] > 1 and x.stride(1) != 1):
        raise ValueError("dropout: x must be a 2-D fp32 tensor with unit column stride")
    rows, n = x.shape
    if out is None:
        out = torch.empty((rows, n), dtype=torch.float32, device=x.device)
    elif out.shape != x.shape or out.dtype != torch.float32 or (n > 1 and out.stride(1) != 1):
        raise ValueError("dropout: bad `out`")
    if rows == 0 or n == 0:
        return out
    seed = _seed_tensor(seed, x.device)
    call("lpf_dropout", ptr(x), max(x.stride(0), n), ptr(out), max(out.stride(0), n), rows, n, int(row0), ptr(seed),
         int(site), float(p), stream(), meta=(rows, n))
    return out


def dropout_mask(seed, site, rows, n, p, row0=0, device="cuda"):
    """The [rows, n] mask of (seed, site) for rows row0 .. row0 + rows, times 1 / (1 - p): lpf_dropout applied to ones
    (the inspection hook of the tests)."""
    dev = seed.device if torch.is_tensor(seed) else torch.device(device)
    return dropout(torch.ones((rows, n), dtype=torch.float32, device=dev), p, seed, site, row0=row0)


def drop_pairs(sel: Selection, p, seed, site=SITE_NODE) -> Selection:
    """Node dropout of a selection (reference drop_pairwise): keeps exactly K = ceil(S (1 - p)) of its S pairs, a uniform
    K-subset drawn from (seed, site), in their order (lpf_drop_pairs_count / _fill), and rebuilds ptr, bounds and nz.
    One host read (the new bounds and the count of non-empty links)."""
    import math
    check_p(p)
    S, bs = sel.total, sel.bs
    K = math.ceil(S * (1.0 - float(p)))
    if K == S:
        return sel
    dev = sel.ptr.device
    seed = _seed_tensor(seed, dev)
    require_cuda(sel.ptr, sel.node, seed)
    ws = torch.empty(_lib.load().lpf_drop_pairs_workspace_bytes() // 8 + 1, dtype=torch.int64, device=dev)
    counts = torch.empty(3 * bs, dtype=torch.int32, device=dev)
    st = stream()
    call("lpf_drop_pairs_count", ptr(sel.ptr), bs, S, K, ptr(seed), int(site), ptr(counts), ptr(ws), 8 * ws.numel(), st,
         meta=(bs, S), launches=18 if K > 0 else 2)
    p_out = torch.empty(3 * bs + 1, dtype=torch.int64, device=dev)
    scratch = torch.empty(max(1, _lib.load().lpf_scan_scratch_bytes(3 * bs) // 8), dtype=torch.int64, device=dev)
    call("lpf_scan_counts", ptr(counts), 3 * bs, ptr(p_out), ptr(scratch), st)
    nz = torch.empty(bs, dtype=torch.int32, device=dev)
    header = torch.empty(4, dtype=torch.int64, device=dev)
    call("lpf_select_compact", ptr(p_out), bs, ptr(nz), ptr(header), st)
    b = header.tolist()          # (S_cn, S_cn + S_1hop, K, #non-empty links)
    if b[2] != K:
        raise _lib.LpfError(f"node dropout kept {b[2]} pairs instead of {K}")
    node = torch.empty(K, dtype=torch.int32, device=dev)
    pa = torch.empty(K, dtype=torch.float32, device=dev)
    pb = torch.empty(K, dtype=torch.float32, device=dev)
    link = torch.empty(K, dtype=torch.int32, device=dev) if sel.link is not None else None
    if K > 0:
        call("lpf_drop_pairs_fill", ptr(sel.ptr), bs, ptr(sel.node), ptr(sel.src_ppr), ptr(sel.tgt_ppr), ptr(sel.link),
             S, ptr(seed), int(site), ptr(ws), ptr(p_out), ptr(node), ptr(pa), ptr(pb), ptr(link), st, meta=(bs, K))
    return Selection(sel.mode, bs, p_out, node, pa, pb, link, (0, b[0], b[1], b[2]), nz[:b[3]])
