"""CPU tests of top-k target retrieval: argument validation of lpf_expand_source_sweep and lpf_topk_fold, the shape and
dtype checks of their ops wrappers, no CPU fallback, evaluate_mrr unchanged on the committed eval goldens after the
rank -> metrics step moved into ranking_metrics, and a world_size-2 gloo test of top_targets_sharded."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from lpformer_b200.build import build
    build()
    from lpformer_b200 import _lib
    return _lib.load()


def test_expand_source_sweep_argument_validation(lib):
    import ctypes as C
    word = C.c_int64(0)
    buf = (C.c_int64 * 8)()
    p = C.addressof(buf)          # any non-NULL pointer: every call below is rejected before a launch
    for s, lk, bad in ((None, p, p), (p, None, p), (p, p, None)):
        assert lib.lpf_expand_source_sweep(s, 4, 3, 0, 4, 10, lk, 4, bad, None) == -1
        assert b"NULL" in lib.lpf_last_error()
    for w in (0, 2, 16):
        assert lib.lpf_expand_source_sweep(p, w, 3, 0, 4, 10, p, 4, p, None) == -1
        assert b"id_bytes" in lib.lpf_last_error()
    assert lib.lpf_expand_source_sweep(p, 4, 0, 0, 4, 10, p, 4, p, None) == -1          # n_targets < 1
    assert lib.lpf_expand_source_sweep(p, 8, 3, 3, 4, 10, p, 4, p, None) == -1          # j0 == n_targets
    assert lib.lpf_expand_source_sweep(p, 8, 3, -1, 4, 10, p, 4, p, None) == -1         # j0 < 0
    assert b"j0" in lib.lpf_last_error()
    assert lib.lpf_expand_source_sweep(p, 8, 11, 0, 4, 10, p, 4, p, None) == -1         # targets past num_nodes
    assert lib.lpf_expand_source_sweep(p, 8, 3, 0, 4, 10, p, 3, p, None) == -1          # ld < n
    # n == 0 is a no-op, even with NULL pointers
    assert lib.lpf_expand_source_sweep(None, 4, 3, 0, 0, 10, None, 0, None, None) == 0
    assert lib.lpf_expand_source_sweep(None, 8, 1, 0, 0, 1, None, 0, C.addressof(word), None) == 0
    assert word.value == 0


def test_topk_fold_argument_validation(lib):
    import ctypes as C
    buf = (C.c_int64 * 8)()
    p = C.addressof(buf)
    ws = lib.lpf_topk_fold_workspace_bytes(1000, 10, 300)
    assert ws > 0 and lib.lpf_topk_fold_workspace_bytes(2000, 10, 300) > ws
    for k in (0, 1025, -3):
        assert lib.lpf_topk_fold_workspace_bytes(1000, k, 300) == -1

    def fold(prob=p, lo=0, n=100, source=p, positive=None, id_bytes=4, Q=1, nt=300, rowptr=None, col=None,
             rows=0, pos_score=None, k=10, key=p, ids=p, ge=None, gt=None, skip=None, work=p, work_bytes=ws):
        return lib.lpf_topk_fold(prob, lo, n, source, positive, id_bytes, Q, nt, rowptr, col, rows, pos_score, k, key,
                                 ids, ge, gt, skip, work, work_bytes, None)

    for k in (0, 1025):
        assert fold(k=k) == -1
        assert b"k must be" in lib.lpf_last_error()
    for w in (0, 2):
        assert fold(id_bytes=w) == -1
        assert b"id_bytes" in lib.lpf_last_error()
    for kw in (dict(prob=None), dict(source=None), dict(key=None), dict(ids=None), dict(work=None)):
        assert fold(**kw) == -1
        assert b"NULL" in lib.lpf_last_error()
    assert fold(positive=p) == -1                                  # positive without its score and counters
    assert fold(rowptr=p) == -1                                    # rowptr without col
    assert fold(lo=250, n=100) == -1                               # past the last query
    assert fold(lo=-1) == -1
    assert fold(nt=0) == -1
    assert fold(work_bytes=lib.lpf_topk_fold_workspace_bytes(100, 10, 300) - 1) == -1
    assert b"workspace" in lib.lpf_last_error()
    # n == 0 is a no-op, even with NULL pointers
    assert fold(prob=None, n=0, source=None, key=None, ids=None, work=None, work_bytes=0) == 0


def test_ops_shape_and_dtype_checks():
    from lpformer_b200 import ops
    from lpformer_b200._lib import LpfError
    src = torch.zeros(3, dtype=torch.int64)
    links = torch.empty((2, 12), dtype=torch.int64)
    bad = torch.zeros(1, dtype=torch.int64)
    with pytest.raises(ValueError):
        ops.expand_source_sweep(src.float(), 4, 0, 12, 10, links, bad)                  # not integer ids
    with pytest.raises(ValueError):
        ops.expand_source_sweep(src.reshape(3, 1), 4, 0, 12, 10, links, bad)            # not 1-D
    with pytest.raises(ValueError):
        ops.expand_source_sweep(src, 4, 0, 13, 10, links, bad)                          # links too short
    with pytest.raises(ValueError):
        ops.expand_source_sweep(src, 4, 1, 12, 10, links, bad)                          # needs a 4th source
    with pytest.raises(LpfError):                                                       # well-formed, on the CPU
        ops.expand_source_sweep(src, 4, 0, 12, 10, links, bad)
    Q, k, N = 3, 5, 40
    ok = dict(prob=torch.zeros(20), lo=0, source=src, n_targets=N, k=k, top_key=torch.zeros(Q, k),
              top_id=torch.zeros(Q, k, dtype=torch.int32), workspace=torch.empty(64, dtype=torch.uint8))
    pos = dict(positive=src.clone(), pos_score=torch.zeros(Q), cnt_ge=torch.zeros(Q, dtype=torch.int64),
               cnt_gt=torch.zeros(Q, dtype=torch.int64))
    for bad_kw in (dict(prob=torch.zeros(20, dtype=torch.float64)), dict(k=0), dict(k=1025),
                   dict(top_key=torch.zeros(Q, k + 1)), dict(top_id=torch.zeros(Q, k, dtype=torch.int64)),
                   dict(source=src.float())):
        with pytest.raises(ValueError):
            ops.topk_fold(**{**ok, **bad_kw})
    with pytest.raises(ValueError):
        ops.topk_fold(**ok, positive=src.clone())                                       # without score and counters
    with pytest.raises(ValueError):
        ops.topk_fold(**ok, **{**pos, "positive": src.int()})                           # dtype differs from source
    with pytest.raises(ValueError):
        ops.topk_fold(**ok, **{**pos, "cnt_ge": torch.zeros(Q, dtype=torch.int32)})
    with pytest.raises(LpfError):                                                       # well-formed, on the CPU
        ops.topk_fold(**ok, **pos)
    with pytest.raises(ValueError):
        ops.topk_fold_workspace(10, 2000, N, "cpu")                                     # k > 1024


def test_top_targets_has_no_cpu_fallback():
    import lpformer_b200 as L
    from oracle.golden import Golden
    from lpformer_b200._lib import LpfError
    from lpformer_b200.evaluate import LinkScoreStream
    g = Golden("all_d32")
    model = L.LinkTransformer(g.train_args(), g.data_dict(), device="cpu").eval()
    score = L.mlp_score(model.out_dim, model.out_dim, 1, 2).eval()
    with pytest.raises((LpfError, RuntimeError, AssertionError)):
        LinkScoreStream(model, score, torch.from_numpy(g["X_node"]), 64).top_targets(torch.arange(4), 3)


def test_evaluate_mrr_unchanged_on_eval_goldens():
    """On the committed citation2-style and HeaRT-style predictions, evaluate_mrr is ranking_metrics of
    get_ranking_list and equals the Hits / MRR formula of the reference, written out here."""
    from lpformer_b200.evaluate import evaluate_mrr, get_ranking_list, ranking_metrics
    z = np.load(os.path.join(REPO, "tests", "golden", "eval", "eval_testset_d32.npz"), allow_pickle=True)
    pos = torch.from_numpy(z["c2_pred_test_pos"])
    neg = torch.from_numpy(z["c2_pred_test_neg"])
    got = evaluate_mrr(pos, neg)
    assert got == ranking_metrics(get_ranking_list(pos, neg))
    rank = get_ranking_list(pos, neg)
    want = [float((rank <= 10).float().mean()), float((rank <= 50).float().mean()),
            float((rank <= 100).float().mean()), float((1.0 / rank).mean())]
    assert [got["Hits@10"], got["Hits@50"], got["Hits@100"], got["MRR"]] == want
    heart_pos = torch.from_numpy(z["plain_pred_test_pos"])
    heart_neg = torch.from_numpy(z["heart_pred_test_neg"])
    assert evaluate_mrr(heart_pos, heart_neg) == ranking_metrics(get_ranking_list(heart_pos, heart_neg))


class _StubStream:
    """Stands in for LinkScoreStream: 'top targets' of a source are a deterministic function of it, tagged with the
    rank that computed them."""

    def __init__(self, rank):
        self.rank, self.seen = rank, []

    def top_targets(self, source, k, exclude=None, positive=None):
        from lpformer_b200.evaluate import TopTargets
        self.seen.append(source.clone())
        s = source.double()[:, None]
        j = torch.arange(k, dtype=torch.float64)[None, :]
        rank = None if positive is None else positive.float() * 0.5 + 0.25 * self.rank
        return TopTargets((s * 0.001 - j * 1e-5).float() + 0.25 * self.rank, (s * 100 + j).long(), rank)


def _worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from lpformer_b200.evaluate import evaluate_full_ranking, ranking_metrics, shard_bounds, top_targets_sharded
        Q, k = 7, 4                                         # 7 queries over 2 ranks: shards of 4 and 3 (padding)
        src = torch.tensor([5, 0, 9, 2, 7, 3, 11], dtype=torch.int32)
        pos = torch.tensor([1, 4, 6, 8, 10, 12, 14])
        bounds = shard_bounds(Q, world)
        owner = torch.zeros(Q)
        for r in range(world):
            owner[bounds[r]:bounds[r + 1]] = r
        for positive in (None, pos):
            st = _StubStream(rank)
            out = top_targets_sharded(None, None, src, None, k, positive=positive, stream=st)
            lo, hi = bounds[rank], bounds[rank + 1]
            assert len(st.seen) == 1 and torch.equal(st.seen[0], src[lo:hi])       # each rank sweeps its own queries
            s = src.double()[:, None]
            j = torch.arange(k, dtype=torch.float64)[None, :]
            assert out.scores.dtype == torch.float32 and out.targets.dtype == torch.int64
            assert torch.equal(out.scores, (s * 0.001 - j * 1e-5).float() + 0.25 * owner[:, None])
            assert torch.equal(out.targets, (s * 100 + j).long())
            if positive is None:
                assert out.rank is None
            else:
                assert torch.equal(out.rank, pos.float() * 0.5 + 0.25 * owner)
        m = evaluate_full_ranking(None, None, src, pos, None, stream=_StubStream(rank))
        assert m == ranking_metrics(pos.float() * 0.5 + 0.25 * owner)
        ret[rank] = True
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_top_targets_sharding_world2_gloo():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(2, port, ret), nprocs=2, join=True)
    assert ret.get(0) and ret.get(1)
