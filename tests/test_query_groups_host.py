"""CPU tests of the query-group input (one source, K targets per query): argument validation of
lpf_expand_query_links, no CPU fallback of score_queries, and a world_size-2 gloo test of score_queries_sharded."""
import os
import socket
from types import SimpleNamespace

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle.golden import Golden


@pytest.fixture(scope="module")
def lib():
    from lpformer_b200.build import build
    build()
    from lpformer_b200 import _lib
    return _lib.load()


def test_expand_query_links_argument_validation(lib):
    import ctypes as C
    word = C.c_int64(0)
    buf = (C.c_int64 * 8)()
    p = C.addressof(buf)          # any non-NULL pointer: every call below is rejected before a launch
    # NULL pointers
    for args in ((None, p, p, p), (p, None, p, p), (p, p, None, p), (p, p, p, None)):
        s, t, lk, bad = args
        assert lib.lpf_expand_query_links(s, t, 4, 3, 0, 4, 10, lk, 4, bad, None) == -1
        assert b"NULL" in lib.lpf_last_error()
    # id width other than int32 / int64
    for w in (0, 2, 16):
        assert lib.lpf_expand_query_links(p, p, w, 3, 0, 4, 10, p, 4, p, None) == -1
        assert b"id_bytes" in lib.lpf_last_error()
    # K < 1, and j0 outside [0, K)
    assert lib.lpf_expand_query_links(p, p, 4, 0, 0, 4, 10, p, 4, p, None) == -1
    assert b"K" in lib.lpf_last_error()
    assert lib.lpf_expand_query_links(p, p, 8, 3, 3, 4, 10, p, 4, p, None) == -1
    assert lib.lpf_expand_query_links(p, p, 8, 3, -1, 4, 10, p, 4, p, None) == -1
    # a leading dimension that cannot hold the range
    assert lib.lpf_expand_query_links(p, p, 8, 3, 0, 4, 10, p, 3, p, None) == -1
    # n == 0 is a no-op, even with NULL pointers
    assert lib.lpf_expand_query_links(None, None, 4, 3, 0, 0, 10, None, 0, None, None) == 0
    assert lib.lpf_expand_query_links(None, None, 8, 1, 0, 0, 0, None, 0, C.addressof(word), None) == 0
    assert word.value == 0


def test_query_groups_shape_and_dtype_checks():
    from lpformer_b200 import ops
    s = torch.zeros(3, dtype=torch.int64)
    ok = ops.query_groups(s, torch.zeros((3, 5), dtype=torch.int64))
    assert ok[0].shape == (3,) and ok[1].shape == (3, 5)
    with pytest.raises(ValueError):
        ops.query_groups(s, torch.zeros(15, dtype=torch.int64))                   # targets not [Q, K]
    with pytest.raises(ValueError):
        ops.query_groups(s, torch.zeros((4, 5), dtype=torch.int64))               # Q mismatch
    with pytest.raises(ValueError):
        ops.query_groups(s, torch.zeros((3, 5), dtype=torch.int32))               # mixed widths
    with pytest.raises(ValueError):
        ops.query_groups(s.float(), torch.zeros((3, 5)))                          # not integer ids


def test_score_queries_has_no_cpu_fallback():
    import lpformer_b200 as L
    from lpformer_b200 import ops
    from lpformer_b200._lib import LpfError
    g = Golden("all_d32")
    model = L.LinkTransformer(g.train_args(), g.data_dict(), device="cpu").eval()
    score = L.mlp_score(model.out_dim, model.out_dim, 1, 2).eval()
    src, tgt = torch.arange(4), torch.arange(12).reshape(4, 3)
    with pytest.raises(LpfError):
        model.score_queries(src, tgt, torch.from_numpy(g["X_node"]), score)
    with pytest.raises(LpfError):
        ops.expand_query_links(src, tgt.reshape(-1), 3, 0, 12, 100, torch.empty((2, 12), dtype=torch.int64),
                               torch.zeros(1, dtype=torch.int64))


def test_query_group_cost_equals_link_group_cost_of_the_pairs():
    import lpformer_b200 as L
    from lpformer_b200.evaluate import link_group_cost, query_group_cost
    g = Golden("all_d32")
    model = L.LinkTransformer(g.train_args(), g.data_dict(), device="cpu").eval()
    n = model.get_adj(False, mask=True).n
    gen = torch.Generator().manual_seed(4)
    Q, K = 9, 6
    src = torch.randint(0, n, (Q,), generator=gen)
    tgt = torch.randint(0, n, (Q, K), generator=gen)
    pairs = torch.stack((src.repeat_interleave(K), tgt.reshape(-1)))
    want = link_group_cost(model, pairs, K)
    assert torch.equal(query_group_cost(model, src, tgt), want)
    assert torch.equal(query_group_cost(model, src.int(), tgt.int()), want)


class _StubModel:
    """Stands in for LinkTransformer: the 'score' of link (a, b) is a deterministic function of (a, b), tagged with the
    rank that computed it; rowptr-only tables give the cost model something to balance."""

    def __init__(self, rank, rowptr):
        self.rank = rank
        self.seen = []
        self.tab = SimpleNamespace(rowptr=rowptr)

    def _dev(self):
        return torch.device("cpu")

    def get_adj(self, test_set=False, mask=False):
        return self.tab

    def get_ppr(self, test_set=False):
        return self.tab

    def score_queries(self, source, targets, X, score_func, test_set=False):
        assert source.dim() == 1 and targets.shape[0] == source.shape[0]
        self.seen.append(source.clone())
        return (source[:, None].double() * 1000 + targets).float() + 0.25 * self.rank


def _worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from lpformer_b200.evaluate import query_group_cost, score_queries_sharded, shard_bounds
        Q, K = 7, 5                                        # 7 queries of 5 links: uneven over 2 ranks
        deg = torch.tensor([0, 1, 9, 2, 400, 3, 0, 1, 5, 2, 7])          # node 4: a hub
        rowptr = torch.cat((torch.zeros(1, dtype=torch.int64), torch.cumsum(deg, 0)))
        src = torch.tensor([4, 0, 1, 2, 7, 3, 5], dtype=torch.int32)       # distinct: a source tags its query
        tgt = (torch.arange(Q * K, dtype=torch.int32) % 4).reshape(Q, K)
        # the hub's query weighs as much as the other six: balanced cuts [0, 1, 7], by count [0, 4, 7]
        assert shard_bounds(Q, world, query_group_cost(_StubModel(rank, rowptr), src, tgt)) != shard_bounds(Q, world)
        model = _StubModel(rank, rowptr)
        for balance in (False, True):
            model.seen = []
            out = score_queries_sharded(model, None, src, tgt, None, batch_size=2 * K + 3, balance=balance)
            bounds = shard_bounds(Q, world, query_group_cost(model, src, tgt) if balance else None)
            lo, hi = bounds[rank], bounds[rank + 1]
            # every query scored once, by its owner, in batches of whole queries (2 per call here)
            seen = torch.cat(model.seen) if model.seen else torch.empty(0, dtype=torch.int32)
            assert torch.equal(seen, src[lo:hi]), (balance, seen, src[lo:hi])
            assert all(s.numel() <= 2 for s in model.seen)
            owner = torch.zeros(Q)
            for r in range(world):
                owner[bounds[r]:bounds[r + 1]] = r
            expect = (src[:, None].double() * 1000 + tgt).float() + 0.25 * owner[:, None]
            assert out.shape == (Q, K) and torch.equal(out, expect)
        ret[rank] = True
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_query_sharding_world2_gloo():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(2, port, ret), nprocs=2, join=True)
    assert ret.get(0) and ret.get(1)
