"""-m gpu: top-k target retrieval over all nodes through every layer — lpf_expand_source_sweep alone, lpf_topk_fold
alone (bit-exact against a stable sort of the materialised candidates), LinkScoreStream.top_targets against the
materialised scores of score_grouped on the plan path, the host-sized path and through pair-pool overflows, and
(>= 2 GPUs) top_targets_sharded under NCCL."""
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-5, 1e-7          # the tolerance of the plan tests (fused / batched regimes differ in fp32 summation order)


def setup(dim=64, seed=5):
    import lpformer_b200 as L
    from lpformer_b200 import synthetic as S
    g = S.make_graph("citation2", seed=seed, scale=0.02, heldout=64)
    cfg = dict(g.cfg, dim=dim)
    dev = torch.device("cuda:0")
    torch.manual_seed(3)
    model = L.LinkTransformer(S.train_args_of(cfg), g.data_dict(dev), device=dev).to(dev).eval()
    score = L.mlp_score(model.out_dim, model.out_dim, 1, 2).to(dev).eval()
    X = torch.randn(g.n, dim, generator=torch.Generator().manual_seed(1)).to(dev)
    return g, model, score, X


# ------------------------------------------------------------------------------------------------------------------
# lpf_expand_source_sweep
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.int32, torch.int64])
@pytest.mark.parametrize("nt", [1, 7, 5003])
def test_sweep_expand_kernel_matches_torch(dtype, nt):
    from lpformer_b200 import ops
    dev = torch.device("cuda:0")
    n_nodes, Q = 50_000, 13
    src = torch.randint(0, n_nodes, (Q,), generator=torch.Generator().manual_seed(nt)).to(dtype).to(dev)
    ref = torch.stack((src.long().repeat_interleave(nt), torch.arange(nt, device=dev).repeat(Q)))
    L = Q * nt
    bad = torch.zeros(1, dtype=torch.int64, device=dev)
    # whole form, then ranges that start inside a query and straddle several (j0 != 0), into a wider buffer
    for lo, hi in ((0, L), (nt // 2, L - 1), (3 * nt + nt - 1, min(L, 7 * nt + 2)), (L - 1, L), (5, 5 + min(L - 5, 2 * nt + 3))):
        n = hi - lo
        q0 = lo // nt
        out = torch.full((2, n + 13), -7, dtype=torch.int64, device=dev)
        ops.expand_source_sweep(src[q0:], nt, lo - q0 * nt, n, n_nodes, out, bad)
        assert torch.equal(out[:, :n], ref[:, lo:hi]), (lo, hi)
        assert bool((out[:, n:] == -7).all())                 # nothing past the range
    assert int(bad.item()) == 0
    # out-of-range sources (-1 and num_nodes) come out as 0 and raise the flag; the targets are untouched
    src2 = src.clone()
    src2[1], src2[Q - 1] = -1, n_nodes
    out = torch.empty((2, L), dtype=torch.int64, device=dev)
    ops.expand_source_sweep(src2, nt, 0, L, n_nodes, out, bad)
    assert int(bad.item()) == 1
    want = ref.clone()
    want[0, nt:2 * nt] = 0
    want[0, (Q - 1) * nt:] = 0
    assert torch.equal(out, want)


# ------------------------------------------------------------------------------------------------------------------
# lpf_topk_fold alone, bit-exact
# ------------------------------------------------------------------------------------------------------------------
def ref_fold(S, src, k, ex_rows, pos=None, pos_score=None):
    """Torch reference on the materialised scores S [Q, N]: candidates = every j but the source and its exclusion row,
    sorted stably by (-score, id); ranks by get_ranking_list over the candidates minus the positive."""
    from lpformer_b200.evaluate import get_ranking_list
    Q, N = S.shape
    keys = torch.full((Q, k), float("-inf"))
    ids = torch.full((Q, k), -1, dtype=torch.int32)
    ranks = torch.zeros(Q)
    for q in range(Q):
        s = int(src[q])
        valid = torch.ones(N, dtype=torch.bool)
        valid[s] = False
        valid[ex_rows.get(s, [])] = False
        cand = torch.nonzero(valid).reshape(-1)                  # ascending ids
        order = torch.sort(-S[q, cand], stable=True)[1][:k]
        keys[q, :order.numel()] = S[q, cand[order]]
        ids[q, :order.numel()] = cand[order].int()
        if pos is not None:
            neg = valid.clone()
            neg[int(pos[q])] = False
            ranks[q] = get_ranking_list(pos_score[q:q + 1], S[q, neg])[0]
    return keys, ids, ranks


def make_csr(rows, n):
    from lpformer_b200.graph import CSR
    rowptr, col = [0], []
    for r in range(n):
        c = sorted(set(rows.get(r, [])))
        col += c
        rowptr.append(len(col))
    return CSR(torch.tensor(rowptr, dtype=torch.int64).cuda(), torch.tensor(col, dtype=torch.int32).cuda(), None, n)


def fold_all(cuts, S, src, k, csr, pos, pos_score, skip=None):
    from lpformer_b200 import ops
    Q, N = S.shape
    dev = torch.device("cuda:0")
    flat = S.reshape(-1).to(dev)
    top_key = torch.full((Q, k), float("-inf"), device=dev)
    top_id = torch.full((Q, k), -1, dtype=torch.int32, device=dev)
    cnt = torch.zeros((2, Q), dtype=torch.int64, device=dev)
    ws = ops.topk_fold_workspace(max(hi - lo for lo, hi in cuts), k, N, dev)
    kw = {}
    if pos is not None:
        kw = dict(positive=pos, pos_score=pos_score, cnt_ge=cnt[0], cnt_gt=cnt[1])
    for lo, hi in cuts:
        ops.topk_fold(flat[lo:hi], lo, src, N, k, top_key, top_id, ws, exclude=csr, skip=skip, **kw)
    return top_key, top_id, cnt


@pytest.mark.parametrize("k", [1, 10, 100, 1024])
@pytest.mark.parametrize("N,Q", [(700, 40), (20_000, 3)])
def test_fold_kernel_bit_exact(k, N, Q):
    """Quantised scores (many ties), n_targets below one tile and far above it, k above the number of candidates
    (padding), exclusion rows (with N = 20,000 one hub row longer than the shared-memory stage), with and without
    positives, two batch cuttings and the reversed order giving identical state, a skipped launch."""
    dev = torch.device("cuda:0")
    gen = torch.Generator().manual_seed(k * 7 + N)
    S = (torch.randint(0, 64, (Q, N), generator=gen).float() / 64.0 - 0.3)      # 64 distinct values: ties everywhere
    src = torch.randperm(N, generator=gen)[:Q]
    src[0] = 3                                                                   # the hub
    ex_rows = {int(s): torch.randint(0, N, (int(torch.randint(0, 40, (1,), generator=gen)),), generator=gen).tolist()
               for s in src[1:]}
    ex_rows[3] = torch.randperm(N, generator=gen)[:min(3000, N // 2)].tolist()
    pos = torch.tensor([(int(s) + 1 + int(torch.randint(0, N - 1, (1,), generator=gen))) % N for s in src])
    pos_score = S[torch.arange(Q), pos] + torch.where(torch.arange(Q) % 2 == 0, 0.0, 1.0 / 128)   # on and between ties
    csr = make_csr(ex_rows, N)
    L = Q * N
    even = [(lo, min(L, lo + 1777)) for lo in range(0, L, 1777)]
    cuts = torch.cumsum(torch.randint(1, 9000, (L // 500 + 2,), generator=gen), 0)
    bounds = [0] + [int(c) for c in cuts if c < L] + [L]
    rev = [(bounds[i], bounds[i + 1]) for i in range(len(bounds) - 1)][::-1]
    for dt in (torch.int64, torch.int32):
        s_dev = src.to(dt).to(dev)
        for with_pos in (False, True):
            p = pos.to(dt).to(dev) if with_pos else None
            ps = pos_score.to(dev) if with_pos else None
            want_k, want_i, want_r = ref_fold(S, src, k, ex_rows, pos if with_pos else None, pos_score)
            a = fold_all(even, S, s_dev, k, csr, p, ps)
            b = fold_all(rev, S, s_dev, k, csr, p, ps)
            for x, y in zip(a, b):
                assert torch.equal(x, y)
            assert torch.equal(a[0].cpu(), want_k)
            assert torch.equal(a[1].cpu(), want_i)
            if with_pos:
                rank = 0.5 * (a[2][0] + a[2][1]).float() + 1
                assert torch.equal(rank.cpu(), want_r)
    # without exclusion: only the source is left out
    no_ex = ref_fold(S, src, k, {})
    got = fold_all(even, S, src.to(dev), k, None, None, None)
    assert torch.equal(got[0].cpu(), no_ex[0]) and torch.equal(got[1].cpu(), no_ex[1])
    # a set skip word: nothing is folded
    skip = torch.ones(1, dtype=torch.int64, device=dev)
    got = fold_all(even, S, src.to(dev), k, csr, pos.to(dev), pos_score.to(dev), skip=skip)
    assert bool((got[0] == float("-inf")).all()) and bool((got[1] == -1).all()) and int(got[2].abs().sum()) == 0


# ------------------------------------------------------------------------------------------------------------------
# LinkScoreStream.top_targets end to end
# ------------------------------------------------------------------------------------------------------------------
def check_top(res, S, src, k, ex, pos=None, pos_score=None):
    """res against the materialised scores S [Q, N] at the plan tolerance: returned scores are those of their links,
    no other candidate beats the k-th returned by more than the tolerance, ranks within the tied window."""
    Q, N = S.shape
    assert res.scores.shape == (Q, k) and res.targets.shape == (Q, k) and res.targets.dtype == torch.int64
    sc, tg = res.scores.cpu(), res.targets.cpu()
    S = S.cpu()
    for q in range(Q):
        s = int(src[q])
        valid = torch.ones(N, dtype=torch.bool)
        valid[s] = False
        if ex is not None:
            valid[ex.col[ex.rowptr[s]:ex.rowptr[s + 1]].long().cpu()] = False
        n_cand = int(valid.sum())
        got = tg[q, :min(k, n_cand)]
        assert bool((tg[q, min(k, n_cand):] == -1).all())
        assert len(set(got.tolist())) == got.numel() and bool(valid[got].all())
        np.testing.assert_allclose(sc[q, :got.numel()].numpy(), S[q, got].numpy(), rtol=RTOL, atol=ATOL)
        assert bool((sc[q, 1:got.numel()] <= sc[q, :got.numel() - 1]).all())            # ordered
        rest = valid.clone()
        rest[got] = False
        if bool(rest.any()):
            kth = float(sc[q, got.numel() - 1])
            assert float(S[q, rest].max()) <= kth + ATOL + RTOL * abs(kth), q
        if pos is not None:
            p, ps = int(pos[q]), float(pos_score[q])
            neg = valid.clone()
            neg[p] = False
            want = 1 + 0.5 * (float((S[q, neg] >= ps).sum()) + float((S[q, neg] > ps).sum()))
            tol = 2 * (ATOL + RTOL * abs(ps))
            window = int(((S[q, neg] - ps).abs() <= tol).sum())
            assert abs(float(res.rank[q]) - want) <= window, (q, float(res.rank[q]), want, window)


def materialised(model, score, X, src, bs, test_set, logits):
    from lpformer_b200.evaluate import LinkScoreStream
    st = LinkScoreStream(model, score, X, bs, test_set=test_set, return_logits=logits, depth=2)
    N = st.num_nodes
    return st.score_grouped(src.cuda(), torch.arange(N).expand(src.numel(), N).contiguous().cuda()), st


@pytest.mark.parametrize("dim", [64, 128])
def test_top_targets_matches_materialised_scores(dim):
    """d = 64 takes the plan path, d = 128 the host-sized one; batches of 2.5 queries + 37 links straddle queries and
    hold several; with and without exclusion, probabilities and logits, the train and the test_set tables, int32 and
    int64 ids from the device and from host memory."""
    from lpformer_b200.evaluate import LinkScoreStream
    g, model, score, X = setup(dim)
    N = model._id_bound(X, False)
    Q, k = 5, 50
    src = torch.from_numpy(g.heldout[0, :Q].copy())
    pos = torch.from_numpy(g.heldout[1, :Q].copy())
    bs = 5 * N // 2 + 37
    ex = model.get_adj(False, mask=True)
    for test_set, logits, exclude in ((False, False, None), (False, True, ex), (True, False, ex), (True, True, None)):
        S, _ = materialised(model, score, X, src, bs, test_set, logits)
        st = LinkScoreStream(model, score, X, bs, test_set=test_set, return_logits=logits, depth=2)
        assert (st.plans is not None) == (dim == 64)
        ps = st.score(torch.stack((src, pos)).cuda())
        for s_in, p_in in ((src.cuda(), pos.cuda()), (src.int(), pos.int())):
            res = st.top_targets(s_in, k, exclude=exclude, positive=p_in)
            check_top(res, S, src, k, exclude, pos, ps.cpu())
        res = st.top_targets(src.cuda(), k, exclude=exclude)
        assert res.rank is None
        check_top(res, S, src, k, exclude)


def test_top_targets_bad_ids_raise():
    from lpformer_b200._lib import LpfError
    from lpformer_b200.evaluate import LinkScoreStream
    g, model, score, X = setup()
    st = LinkScoreStream(model, score, X, 50_000, depth=2)
    N = st.num_nodes
    src = torch.tensor([1, 2, 3]).cuda()
    for s, p in ((torch.tensor([1, N, 3]), None), (src, torch.tensor([5, 2, 7])), (src, torch.tensor([5, -1, 7]))):
        with pytest.raises(LpfError):
            st.top_targets(s.cuda(), 4, positive=None if p is None else p.cuda())
    with pytest.raises(ValueError):
        st.top_targets(src, 0)


def test_top_targets_through_pool_overflows():
    """Plans with pair pools of 2 rows: nearly every batch overflows, its fold is skipped on the device and the batch
    is folded when it is re-scored; the result still satisfies the checks against the materialised scores."""
    from lpformer_b200.evaluate import LinkScoreStream
    g, model, score, X = setup()
    N = model._id_bound(X, False)
    Q, k = 4, 100
    src = torch.from_numpy(g.heldout[0, :Q].copy())
    pos = torch.from_numpy(g.heldout[1, :Q].copy())
    bs = 3 * N // 2 + 11
    ex = model.get_adj(False, mask=True)
    S, _ = materialised(model, score, X, src, bs, False, False)
    st = LinkScoreStream(model, score, X, bs, depth=2)
    ps = st.score(torch.stack((src, pos)).cuda()).cpu()
    for P in st.plans:
        P.__init__(P.model, P.score_func, P.consts, P.X, P.kv, P.bs, P.test_set, P.logits, cap=2, use_graph=P.use_graph)
    res = st.top_targets(src.cuda(), k, exclude=ex, positive=pos.cuda())
    assert st.plans[0].cap > 2
    check_top(res, S, src, k, ex, pos, ps)


# ------------------------------------------------------------------------------------------------------------------
# top_targets_sharded under NCCL
# ------------------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out):
    import torch.distributed as dist
    from lpformer_b200.evaluate import LinkScoreStream, top_targets_sharded
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    import lpformer_b200 as L
    from lpformer_b200 import synthetic as S
    g = S.make_graph("citation2", seed=21, scale=0.02, heldout=64)
    torch.manual_seed(3)
    model = L.LinkTransformer(S.train_args_of(g.cfg), g.data_dict(dev), device=dev).to(dev).eval()
    score = L.mlp_score(model.out_dim, model.out_dim, 1, 2).to(dev).eval()
    X = model.propagate()
    src = torch.from_numpy(g.heldout[0, :5].copy())
    pos = torch.from_numpy(g.heldout[1, :5].copy())
    ex = model.get_adj(False, mask=True)
    bs = model._id_bound(X, False)                 # one query per batch on every rank
    got = top_targets_sharded(model, score, src, X, 20, exclude=ex, positive=pos, batch_size=bs)
    one = LinkScoreStream(model, score, X, bs).top_targets(src, 20, exclude=ex, positive=pos)
    if rank == 0:
        out["shape"] = tuple(got.scores.shape)
        out["targets"] = bool(torch.equal(got.targets, one.targets))
        out["scores"] = float((got.scores - one.scores).abs().max())
        out["rank"] = float((got.rank - one.rank).abs().max())
    dist.barrier()
    dist.destroy_process_group()


def test_top_targets_sharded_two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
        assert out["shape"] == (5, 20)
        # (a plan's regime may differ between the runs: scores equal at the plan tolerance)
        assert out["targets"] and out["scores"] <= 1e-6 and out["rank"] <= 1.0, dict(out)
