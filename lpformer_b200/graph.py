"""HBM-resident graph tables consumed by the kernels.

The reference keeps `adj_mask` / `ppr` as N x N torch sparse COO tensors and `adj_t` as a
torch_sparse.SparseTensor (reference util/read_datasets.py:85-129) and slices rows with
sparse index_select on every batch.  Here each table is converted ONCE into a sorted CSR
(rowptr int64 [N+1], col int32 [nnz] ascending per row, val fp32 [nnz]) living in HBM; the
kernels address rows directly.  These conversions are one-time set-up and use torch ops.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import torch


@dataclass
class CSR:
    rowptr: torch.Tensor            # int64 [n+1]
    col: torch.Tensor               # int32 [nnz]
    val: Optional[torch.Tensor]     # fp32 [nnz] or None (0/1 mask)
    n: int
    unit_range: Optional[bool] = None   # cached: all values in (0, 1] (lets K1 use its intersection algorithm)

    @property
    def nnz(self) -> int:
        return int(self.col.numel())

    def to(self, device):
        return CSR(self.rowptr.to(device), self.col.to(device), None if self.val is None else self.val.to(device), self.n)

    def nbytes(self) -> int:
        return self.rowptr.numel() * 8 + self.col.numel() * 4 + (0 if self.val is None else self.val.numel() * 4)


def csr_from_coo(row, col, val, n, device=None, drop_zeros=False) -> CSR:
    """Sorted, duplicate-summed CSR from COO triplets (any order)."""
    row = torch.as_tensor(row, dtype=torch.int64)
    col = torch.as_tensor(col, dtype=torch.int64)
    if device is not None:
        row, col = row.to(device), col.to(device)
    if val is not None:
        val = torch.as_tensor(val, dtype=torch.float32).to(row.device)
    key = row * n + col
    order = torch.argsort(key, stable=True)
    key = key[order]
    if val is not None:
        val = val[order]
    if key.numel() > 1 and bool((key[1:] == key[:-1]).any()):
        # coalesce duplicates (sum), as torch.sparse coalesce() would
        uniq, inv = torch.unique_consecutive(key, return_inverse=True)
        if val is not None:
            val = torch.zeros(uniq.numel(), dtype=val.dtype, device=val.device).index_add_(0, inv, val)
        key = uniq
    if drop_zeros and val is not None:
        keep = val != 0
        key, val = key[keep], val[keep]
    r = torch.div(key, n, rounding_mode="floor")
    c = (key - r * n).to(torch.int32)
    rowptr = torch.zeros(n + 1, dtype=torch.int64, device=key.device)
    rowptr[1:] = torch.cumsum(torch.bincount(r, minlength=n), 0)
    return CSR(rowptr.contiguous(), c.contiguous(), None if val is None else val.contiguous(), n)


def csr_from_sparse(t, device=None, mask=False) -> CSR:
    """CSR from what the reference's `data` dict holds: a torch sparse COO/CSR tensor, a
    torch_sparse.SparseTensor-like object (has .coo()), or an existing CSR.  With
    `mask=True` values are dropped and explicit zeros removed (adj_mask is 0/1,
    reference util/read_datasets.py:95)."""
    if isinstance(t, CSR):
        return t if device is None else t.to(device)
    if hasattr(t, "coo") and not isinstance(t, torch.Tensor):     # torch_sparse.SparseTensor
        row, col, val = t.coo()
        n = t.sparse_sizes()[0]
    elif isinstance(t, torch.Tensor) and t.layout == torch.sparse_csr:
        crow, col, val = t.crow_indices(), t.col_indices(), t.values()
        n = t.shape[0]
        row = torch.repeat_interleave(torch.arange(n, device=crow.device), crow[1:] - crow[:-1])
    elif isinstance(t, torch.Tensor) and t.layout == torch.sparse_coo:
        t = t.coalesce()
        row, col = t.indices()
        val = t.values()
        n = t.shape[0]
    else:
        raise TypeError(f"cannot build a CSR from {type(t)}")
    if mask:
        if val is not None:
            keep = val != 0
            row, col = row[keep], col[keep]
        val = None
    elif val is None:
        val = torch.ones(row.numel(), dtype=torch.float32, device=row.device)
    return csr_from_coo(row, col, None if val is None else val.float(), n, device=device)


def gcn_normalise(adj: CSR) -> CSR:
    """PyG 2.2.0 `gcn_norm` on a SparseTensor (what GCNConv(normalize=True) applies,
    reference models/other_models.py:35-48): missing values = 1, diagonal SET to 1
    (existing self-loops replaced), deg = row sum, A_hat = D^-1/2 A D^-1/2 (inf -> 0)."""
    n, dev = adj.n, adj.rowptr.device
    row = torch.repeat_interleave(torch.arange(n, device=dev), adj.rowptr[1:] - adj.rowptr[:-1])
    col = adj.col.to(torch.int64)
    val = torch.ones(col.numel(), dtype=torch.float32, device=dev) if adj.val is None else adj.val
    keep = row != col
    ar = torch.arange(n, device=dev)
    row = torch.cat([row[keep], ar])
    col = torch.cat([col[keep], ar])
    val = torch.cat([val[keep], torch.ones(n, dtype=torch.float32, device=dev)])
    deg = torch.zeros(n, dtype=torch.float32, device=dev).index_add_(0, row, val)
    dis = deg.pow(-0.5)
    dis[torch.isinf(dis)] = 0.0
    val = dis[row] * val * dis[col]
    return csr_from_coo(row, col, val, n)


def transpose_csr(adj: CSR) -> CSR:
    """The transpose of `adj` (the SpMM of the GCN's backward multiplies by A_hat^T): `adj` itself when it is symmetric
    (every graph gcn_normalise builds from a symmetric adjacency), otherwise a transposed copy.  Either answer is kept on
    the table, so it is worked out once per table."""
    hit = adj.__dict__.get("_transpose")
    if hit is not None:
        return adj if hit is True else hit
    row = torch.repeat_interleave(torch.arange(adj.n, device=adj.rowptr.device), adj.rowptr[1:] - adj.rowptr[:-1])
    t = csr_from_coo(adj.col.to(torch.int64), row, adj.val, adj.n)
    same = bool(torch.equal(t.rowptr, adj.rowptr) and torch.equal(t.col, adj.col) and
                (adj.val is None or torch.equal(t.val, adj.val)))
    adj.__dict__["_transpose"] = True if same else t
    return adj if same else t
