"""-m gpu: query groups (one source, K targets per query) through every layer — lpf_expand_query_links alone,
LinkTransformer.score_queries against score_links, LinkScoreStream.score_grouped against score() on the expanded
links, the citation2 driver, and (>= 2 GPUs) score_queries_sharded under NCCL."""
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def same(x, y):     # the tolerance of the plan tests (fused / batched regimes differ in fp32 summation order)
    np.testing.assert_allclose(x.cpu().numpy(), y.cpu().numpy(), rtol=1e-5, atol=1e-7)


def expand(src, tgt):
    K = tgt.shape[1]
    return torch.stack((src.long().repeat_interleave(K), tgt.long().reshape(-1)))


def setup(dim=64, seed=5, heldout=256):
    import lpformer_b200 as L
    from lpformer_b200 import synthetic as S
    g = S.make_graph("citation2", seed=seed, scale=0.02, heldout=heldout)
    cfg = dict(g.cfg, dim=dim)
    dev = torch.device("cuda:0")
    torch.manual_seed(3)
    model = L.LinkTransformer(S.train_args_of(cfg), g.data_dict(dev), device=dev).to(dev).eval()
    score = L.mlp_score(model.out_dim, model.out_dim, 1, 2).to(dev).eval()
    X = torch.randn(g.n, dim, generator=torch.Generator().manual_seed(1)).to(dev)
    return g, model, score, X


def queries(g, Q, negs, seed):
    """citation2-style groups: the held-out positive then `negs` uniform negatives per source."""
    from lpformer_b200 import synthetic as S
    lk = torch.from_numpy(S.citation2_queries(g, Q, negs, seed=seed))
    K = 1 + negs
    return lk[0, ::K].contiguous(), lk[1].reshape(Q, K).contiguous()


@pytest.mark.parametrize("dtype", [torch.int32, torch.int64])
@pytest.mark.parametrize("K", [1, 7, 1001])
def test_expand_kernel_matches_repeat_interleave(dtype, K):
    from lpformer_b200 import ops
    dev = torch.device("cuda:0")
    n_nodes, Q = 50_000, 37
    gen = torch.Generator().manual_seed(K)
    src = torch.randint(0, n_nodes, (Q,), generator=gen).to(dtype).to(dev)
    tgt = torch.randint(0, n_nodes, (Q, K), generator=gen).to(dtype).to(dev)
    ref = expand(src, tgt)
    flat = tgt.reshape(-1)
    L = Q * K
    bad = torch.zeros(1, dtype=torch.int64, device=dev)
    # whole form, then ranges that start inside a query and straddle several (j0 != 0), into a wider buffer
    for lo, hi in ((0, L), (K // 2, L - 1), (3 * K + K - 1, min(L, 7 * K + 2)), (L - 1, L), (5, 5 + min(L - 5, 2 * K + 3))):
        n = hi - lo
        q0 = lo // K
        out = torch.full((2, n + 13), -7, dtype=torch.int64, device=dev)
        ops.expand_query_links(src[q0:], flat[lo:], K, lo - q0 * K, n, n_nodes, out, bad)
        assert torch.equal(out[:, :n], ref[:, lo:hi]), (lo, hi)
        assert bool((out[:, n:] == -7).all())                 # nothing past the range
    assert int(bad.item()) == 0
    # out-of-range ids (-1 and num_nodes) come out as 0 and raise the flag; the rest is untouched
    src2, tgt2 = src.clone(), tgt.clone()
    src2[1] = -1
    tgt2[2, K - 1] = n_nodes
    out = torch.empty((2, L), dtype=torch.int64, device=dev)
    ops.expand_query_links(src2, tgt2.reshape(-1), K, 0, L, n_nodes, out, bad)
    assert int(bad.item()) == 1
    want = ref.clone()
    want[0, K:2 * K] = 0
    want[1, 2 * K + K - 1] = 0
    assert torch.equal(out, want)


@pytest.mark.parametrize("dim", [64, 32])
def test_score_queries_matches_score_links(dim):
    """d = 64 (fp16-split heads) and d = 32 (3xTF32 heads); the train and the test_set tables; probabilities and logits;
    int32 and int64 ids, on the device and in pinned host memory."""
    from lpformer_b200._lib import LpfError
    g, model, score, X = setup(dim)
    src, tgt = queries(g, 6, 150, seed=11)
    pairs = expand(src, tgt).cuda()
    for test_set in (False, True):
        for logits in (False, True):
            ref = model.score_links(pairs, X, score, test_set=test_set, return_logits=logits).clone()
            for dt in (torch.int64, torch.int32):
                for s, t in ((src.to(dt).cuda(), tgt.to(dt).cuda()), (src.to(dt).pin_memory(), tgt.to(dt).pin_memory())):
                    got = model.score_queries(s, t, X, score, test_set=test_set, return_logits=logits)
                    assert got.shape == tgt.shape
                    same(got.reshape(-1), ref)
    bad_t = tgt.clone().cuda()
    bad_t[0, 3] = g.n
    with pytest.raises(LpfError):
        model.score_queries(src.cuda(), bad_t, X, score)
    same(model.score_queries(src.cuda(), tgt.cuda(), X, score).reshape(-1), model.score_links(pairs, X, score))


def test_score_grouped_matches_score():
    """score_grouped against score() on the expanded links, each on a fresh stream of the same configuration, with a
    batch size that is not a multiple of K (batches straddle queries): device input, pinned host input with out_host,
    a ragged tail, a forced pool overflow (cap = 2) noticed one batch late."""
    from lpformer_b200.evaluate import LinkScoreStream
    g, model, score, X = setup()
    Q, negs = 23, 150
    src, tgt = queries(g, Q, negs, seed=7)
    K = 1 + negs
    pairs = expand(src, tgt)
    bs = 4 * K + 37                                     # 5 full batches + a ragged tail
    assert pairs.shape[1] % bs != 0 and bs % K != 0

    def fresh():
        st = LinkScoreStream(model, score, X, bs, depth=2)
        assert st.plans is not None
        return st

    a, b = fresh(), fresh()
    ref = a.score(pairs.cuda())
    for dt in (torch.int64, torch.int32):
        got = b.score_grouped(src.to(dt).cuda(), tgt.to(dt).cuda())
        assert got.shape == (Q, K)
        same(got.reshape(-1), ref)
        host_out = torch.empty(Q * K, dtype=torch.float32).pin_memory()
        got = b.score_grouped(src.to(dt).pin_memory(), tgt.to(dt).pin_memory(), out_host=host_out)
        same(got.reshape(-1), ref)
        assert torch.equal(host_out, got.reshape(-1).cpu())
    # pools of 2 rows per type: every batch with a non-empty link overflows, is noticed late and re-scored
    a, b = fresh(), fresh()
    for st in (a, b):
        for P in st.plans:
            P.__init__(P.model, P.score_func, P.consts, P.X, P.kv, P.bs, P.test_set, P.logits, cap=2, use_graph=P.use_graph)
    ref = a.score(pairs.cuda())
    got = b.score_grouped(src.cuda(), tgt.cuda())
    same(got.reshape(-1), ref)
    assert b.plans[0].cap > 2
    host_out = torch.empty(Q * K, dtype=torch.float32).pin_memory()
    got = b.score_grouped(src.pin_memory(), tgt.pin_memory(), out_host=host_out)
    same(got.reshape(-1), ref)
    assert torch.equal(host_out, got.reshape(-1).cpu())


def test_score_grouped_bad_ids_raise_and_stream_stays_usable():
    from lpformer_b200._lib import LpfError
    from lpformer_b200.evaluate import LinkScoreStream
    g, model, score, X = setup()
    Q, negs = 12, 100
    src, tgt = queries(g, Q, negs, seed=9)
    K = 1 + negs
    bs = 3 * K + 5
    ref = LinkScoreStream(model, score, X, bs, depth=2).score(expand(src, tgt).cuda())
    st = LinkScoreStream(model, score, X, bs, depth=2)
    bad_mid, bad_tail, bad_src = tgt.clone(), tgt.clone(), src.clone()
    bad_mid[4, 7] = -1                               # inside a plan batch
    bad_tail[Q - 1, K - 1] = g.n                     # in the ragged tail (expanded outside the plans)
    bad_src[2] = g.n + 5
    for s, t in ((src, bad_mid), (src, bad_tail), (bad_src, tgt)):
        with pytest.raises(LpfError):
            st.score_grouped(s.cuda(), t.cuda())
        same(st.score_grouped(src.cuda(), tgt.cuda()).reshape(-1), ref)
    with pytest.raises(LpfError):
        st.score_grouped(src.pin_memory(), bad_mid.pin_memory())
    same(st.score_grouped(src.pin_memory(), tgt.pin_memory()).reshape(-1), ref)
    same(st.score(expand(src, tgt).cuda()), ref)      # the pair form on the same stream, after the flags were raised


def test_citation2_driver_scores_query_groups():
    from lpformer_b200.evaluate import test_edge_citation2
    g, model, score, X = setup()
    pos = torch.from_numpy(g.heldout[:, :16].T.copy())
    neg = torch.from_numpy(np.random.default_rng(0).integers(0, g.n, (16, 50)))
    src = pos[:, 0]
    chk = model.score_links(expand(src, neg).cuda(), X, score).view(16, 50)
    for n in (neg, neg.int()):
        pred = test_edge_citation2(model, score, pos, X, 333, mrr_mode=True, negative_data=n)
        assert pred.shape == (16, 50)
        same(pred, chk)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out):
    import torch.distributed as dist
    from lpformer_b200.evaluate import score_queries_sharded
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    import lpformer_b200 as L
    from lpformer_b200 import synthetic as S
    g = S.make_graph("citation2", seed=21, scale=0.02, heldout=128)
    torch.manual_seed(3)
    model = L.LinkTransformer(S.train_args_of(g.cfg), g.data_dict(dev), device=dev).to(dev).eval()
    score = L.mlp_score(model.out_dim, model.out_dim, 1, 2).to(dev).eval()
    X = model.propagate()
    lk = torch.from_numpy(S.citation2_queries(g, 17, 100, seed=5))
    src, tgt = lk[0, ::101].contiguous(), lk[1].reshape(17, 101).contiguous()
    got = score_queries_sharded(model, score, src, tgt, X, batch_size=3 * 101)
    one = model.score_queries(src.to(dev), tgt.to(dev), X, score)
    if rank == 0:
        out["shape"] = tuple(got.shape)
        out["diff"] = float((got - one).abs().max())
    dist.barrier()
    dist.destroy_process_group()


def test_score_queries_sharded_two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
        assert out["shape"] == (17, 101)
        assert out["diff"] <= 1e-6, out["diff"]
