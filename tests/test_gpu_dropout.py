"""-m gpu: dropout of the training path.  The kernels alone (lpf_dropout, the fused GCN epilogue with dropout, node
dropout of a selection), then the whole model with every dropout > 0 against float64 autograd with the same masks and
kept pairs injected (recovered with ops.dropout_mask and compute_node_mask), and the semantics (eval mode, no_grad,
reproducibility from torch.manual_seed)."""
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import ref_port
from oracle.golden import GOLDEN_CASES, Golden

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
GRAD_RTOL = 1e-4
DROPS = dict(feat_drop=0.3, gnn_drop=0.3, dropout=0.3, att_drop=0.25)
PRED_DROP = 0.3


def _close(got, ref, name, rtol=GRAD_RTOL):
    assert got is not None, f"{name}: no gradient"
    got = got.detach().double().cpu()
    ref = ref.detach().double().cpu()
    assert got.shape == ref.shape, (name, got.shape, ref.shape)
    scale = float(ref.abs().max())
    err = float((got - ref).abs().max())
    assert err <= rtol * scale + 1e-12, f"{name}: max abs err {err:.3g} vs max abs {scale:.3g}"


def _seed(v):
    return torch.tensor([v], dtype=torch.int64, device=DEV)


# ------------------------------------------------------------------------------------------------ lpf_dropout alone
def _philox_word(seed, site, row, col):
    """Word col & 3 of Philox4x32-10 (key = seed, counter = (col >> 2, row, row >> 32, site)): the rule of the header."""
    M0, M1, W0, W1, m32 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85, 0xFFFFFFFF
    c = [col >> 2, row & m32, row >> 32, site]
    k0, k1 = seed & m32, (seed >> 32) & m32
    for r in range(10):
        if r:
            k0, k1 = (k0 + W0) & m32, (k1 + W1) & m32
        p0, p1 = M0 * c[0], M1 * c[2]
        c = [((p1 >> 32) ^ c[1] ^ k0) & m32, p1 & m32, ((p0 >> 32) ^ c[3] ^ k1) & m32, p0 & m32]
    return c[col & 3]


def test_masks_follow_the_documented_philox_rule():
    from lpformer_b200 import ops
    p, seed, site = 0.4, 0x0123456789ABCDEF, 33
    m = ops.dropout_mask(_seed(seed), site, 5, 11, p, row0=(1 << 32) - 2).cpu()
    thr = math.floor(p * 2 ** 32)
    for r in range(5):
        for c in range(11):
            keep = _philox_word(seed, site, (1 << 32) - 2 + r, c) >= thr
            assert bool(m[r, c] != 0) == keep, (r, c)


@pytest.mark.parametrize("p", [0.1, 0.5, 0.9])
def test_keep_fraction_and_scale(p):
    from lpformer_b200 import ops
    n = 1 << 24
    x = torch.randn(4096, n // 4096, device=DEV)
    y = ops.dropout(x, p, _seed(11), ops.SITE_FEATURE)
    kept = y != 0
    frac = float(kept.double().mean())
    sigma = math.sqrt(p * (1 - p) / n)
    assert abs(frac - (1 - p)) <= 6 * sigma, (frac, 1 - p)
    scale = torch.tensor(1.0 / (1.0 - p), dtype=torch.float32, device=DEV)
    assert torch.equal(y[kept], x[kept] * scale)
    # two seeds, and two sites of one seed: agreement of the masks ~ (1-p)^2 + p^2
    for other in (ops.dropout_mask(_seed(12), ops.SITE_FEATURE, 4096, n // 4096, p),
                  ops.dropout_mask(_seed(11), ops.SITE_GCN, 4096, n // 4096, p)):
        agree = float(((other != 0) == kept).double().mean())
        q = (1 - p) ** 2 + p ** 2
        assert abs(agree - q) <= 6 * math.sqrt(q * (1 - q) / n), (agree, q)


def test_p0_is_the_identity_and_p1_zeros():
    from lpformer_b200 import ops
    x = torch.randn(1000, 37, device=DEV)
    x[0, 0] = -0.0
    x[1, 1] = float("inf")
    y = ops.dropout(x, 0.0, _seed(3), ops.SITE_ATT)
    assert torch.equal(y.view(torch.int32), x.view(torch.int32))          # bit for bit
    assert not bool(ops.dropout(x, 1.0, _seed(3), ops.SITE_ATT).any())


def test_row0_slices_and_strided_rows():
    from lpformer_b200 import ops
    full = ops.dropout_mask(_seed(5), ops.SITE_GCN + 1, 3000, 70, 0.5)
    assert torch.equal(ops.dropout_mask(_seed(5), ops.SITE_GCN + 1, 1000, 70, 0.5, row0=1234), full[1234:2234])
    big = torch.randn(3000, 100, device=DEV)
    view = big[:, 7:77]
    ref = view * full
    ops.dropout(view, 0.5, _seed(5), ops.SITE_GCN + 1, out=view)        # in place on a strided view
    assert torch.equal(view, ref)


# ------------------------------------------------------------------------------------------ fused GCN epilogue
def _graph(n, deg, seed):
    from lpformer_b200.graph import csr_from_sparse, gcn_normalise
    gen = torch.Generator().manual_seed(seed)
    e = torch.randint(0, n, (2, n * deg), generator=gen)
    e = torch.cat((e, e.flip(0)), 1)
    adj = torch.sparse_coo_tensor(e, torch.ones(e.shape[1]), (n, n)).coalesce()
    return gcn_normalise(csr_from_sparse(adj, DEV))


@pytest.mark.parametrize("d", [32, 64, 128, 256])
@pytest.mark.parametrize("residual,ln2", [(False, False), (True, False), (True, True), (False, True)])
def test_gcn_layer_with_dropout_matches_the_unfused_composition(d, residual, ln2):
    from lpformer_b200 import ops
    torch.manual_seed(d)
    n, p, site = 5003, 0.3, ops.SITE_GCN + 2
    adj = _graph(n, 6, d)
    xw = torch.randn(n, d, device=DEV)
    res = torch.randn(n, d, device=DEV) if residual else None
    b = 0.1 * torch.randn(d, device=DEV)
    ln = (1 + 0.2 * torch.randn(d, device=DEV), 0.1 * torch.randn(d, device=DEV))
    l2 = (1 + 0.2 * torch.randn(d, device=DEV), 0.1 * torch.randn(d, device=DEV)) if ln2 else None
    seed = _seed(77)
    got = ops.gcn_layer(adj, xw, b, ln=ln, relu=True, residual=res, ln2=l2, dropout=(p, seed, site))
    y = ops.gcn_spmm(adj, xw, b)
    m = ops.dropout_mask(seed, site, n, d, p)
    u = F.relu(F.layer_norm(y, (d,), *ln, eps=1e-5)) * m
    if residual:
        u = u + res
    if ln2:
        u = F.layer_norm(u, (d,), *l2, eps=1e-5)
    torch.testing.assert_close(got, u, rtol=1e-5, atol=1e-5)
    # the recompute of the GCN backward (lpf_layernorm_act_dropout) gives the pre-gnn_norm rows of the fused kernel
    pre = ops.layernorm_act(y, *ln, relu=True, residual=res, dropout=(p, seed, site))
    want = ops.gcn_layer(adj, xw, b, ln=ln, relu=True, residual=res, dropout=(p, seed, site))
    torch.testing.assert_close(pre, want, rtol=1e-5, atol=1e-5)
    # p = 0: bit-identical to lpf_gcn_layer; a row range (row0) reads the node-id rows of the full mask
    zero = ops.gcn_layer(adj, xw, b, ln=ln, relu=True, residual=res, ln2=l2, dropout=(0.0, seed, site))
    assert torch.equal(zero, ops.gcn_layer(adj, xw, b, ln=ln, relu=True, residual=res, ln2=l2))
    part = torch.zeros_like(got)
    ops.gcn_layer(adj, xw, b, ln=ln, relu=True, residual=res, ln2=l2, out=part, row0=1000, rows=2000,
                  dropout=(p, seed, site))
    assert torch.equal(part[1000:3000], got[1000:3000])


# ------------------------------------------------------------------------------------------------- node dropout
def _selection(sizes, seed):
    """A Selection of len(sizes) // 3 links with segment sizes `sizes` (type-major): node = the pair's position (a
    payload the kernels only move), random PPR values."""
    from lpformer_b200 import ops
    gen = torch.Generator().manual_seed(seed)
    counts = torch.as_tensor(sizes, dtype=torch.int64)
    bs = counts.numel() // 3
    ptr = torch.zeros(3 * bs + 1, dtype=torch.int64)
    ptr[1:] = torch.cumsum(counts, 0)
    S = int(ptr[-1])
    link = (torch.repeat_interleave(torch.arange(3 * bs), counts) % bs).to(torch.int32)
    bounds = tuple(int(ptr[k * bs]) for k in range(3)) + (S,)
    nz = torch.nonzero(counts.view(3, bs).sum(0) > 0).reshape(-1).to(torch.int32)
    return ops.Selection("all", bs, ptr.to(DEV), torch.arange(S, dtype=torch.int32, device=DEV),
                         torch.rand(S, generator=gen).to(DEV), torch.rand(S, generator=gen).to(DEV), link.to(DEV),
                         bounds, nz.to(DEV))


@pytest.mark.parametrize("S", [0, 1, 50, 10 ** 6, 2 * 10 ** 7])
@pytest.mark.parametrize("p", [0.0, 0.25, 1.0])
def test_node_dropout_keeps_exactly_k_pairs_in_order(S, p):
    from lpformer_b200 import ops
    bs = max(1, min(S // 50, 100000))
    gen = torch.Generator().manual_seed(S)
    w = torch.rand(3 * bs, generator=gen) ** 3
    sizes = torch.floor(w / w.sum() * S).long()
    sizes[0] += S - int(sizes.sum())
    sel = _selection(sizes.tolist(), S)
    K = math.ceil(S * (1 - p))
    out = ops.drop_pairs(sel, p, _seed(S + 1))
    assert out.total == K
    if K == S:
        assert out is sel
        return
    cnt = (out.ptr[1:] - out.ptr[:-1])
    assert int(out.ptr[-1]) == K and bool((cnt >= 0).all()) and bool((cnt <= (sel.ptr[1:] - sel.ptr[:-1])).all())
    assert out.bounds == tuple(int(out.ptr[k * bs]) for k in range(3)) + (K,)
    live = torch.nonzero(cnt.view(3, bs).sum(0) > 0).reshape(-1)
    assert torch.equal(torch.sort(out.nz.long())[0], live)
    if K == 0:
        return
    # order: the kept pairs are a subsequence of the input, each in its input segment, with its payload
    seg_out = torch.repeat_interleave(torch.arange(3 * bs, device=DEV), cnt)
    seg_in = torch.repeat_interleave(torch.arange(3 * bs, device=DEV), sel.ptr[1:] - sel.ptr[:-1])
    idx = out.node.long()                                      # (node holds the input position)
    assert bool((idx[1:] > idx[:-1]).all())
    assert torch.equal(seg_in[idx], seg_out) and torch.equal(out.link.long(), seg_out % bs)
    assert torch.equal(out.src_ppr, sel.src_ppr[idx]) and torch.equal(out.tgt_ppr, sel.tgt_ppr[idx])


def test_node_dropout_is_a_uniform_k_subset():
    from lpformer_b200 import ops
    sel = _selection([5, 0, 12, 3, 9, 0, 7, 10, 4], 3)          # 50 pairs over 3 links
    S, p = 50, 0.3
    K = math.ceil(S * (1 - p))
    draws = 4000
    inc = torch.zeros(S, dtype=torch.float64)
    pairs = [(0, 1), (4, 30), (17, 49), (20, 21)]
    joint = torch.zeros(len(pairs), dtype=torch.float64)
    for i in range(draws):
        out = ops.drop_pairs(sel, p, _seed(1000 + i))
        pos = out.node.long().cpu()                                      # (node holds the input position)
        hit = torch.zeros(S, dtype=torch.float64)
        hit[pos] = 1
        assert int(hit.sum()) == K
        inc += hit
        for j, (a, b) in enumerate(pairs):
            joint[j] += hit[a] * hit[b]
    q = K / S
    sd = math.sqrt(q * (1 - q) / draws)
    assert float((inc / draws - q).abs().max()) <= 4.5 * sd, (inc / draws)
    q2 = K * (K - 1) / (S * (S - 1))
    sd2 = math.sqrt(q2 * (1 - q2) / draws)
    assert float((joint / draws - q2).abs().max()) <= 4.5 * sd2, (joint / draws, q2)


# ------------------------------------------------------------------------------------------ whole model vs float64
def _build(g, **drops):
    import lpformer_b200 as L
    data = g.data_dict(DEV)
    if "emb" in data:
        data["emb"].weight.requires_grad_(True)
    model = L.LinkTransformer(dict(g.train_args(), **drops), data, device=DEV).to(DEV)
    score = L.mlp_score(model.out_dim, model.out_dim, 1, 2, dropout=PRED_DROP if drops else 0).to(DEV)
    msd, ssd = g.state_dicts(DEV)
    model.load_state_dict(msd)
    score.load_state_dict(ssd)
    return model, score


def _dense_ahat(model, adj=None):
    from lpformer_b200.graph import csr_from_sparse, gcn_normalise
    a = model.get_adj(False) if adj is None else gcn_normalise(csr_from_sparse(adj, DEV))
    n = a.n
    row = torch.repeat_interleave(torch.arange(n), (a.rowptr[1:] - a.rowptr[:-1]).cpu())
    return torch.sparse_coo_tensor(torch.stack((row, a.col.long().cpu())), a.val.double().cpu(), (n, n)).to_dense()


def _masks(model, score, bs):
    """Every mask of the last forward, recovered from the modules' seeds (values mask / (1 - p), float64)."""
    from lpformer_b200 import ops
    enc = model.node_encoder
    gcn = enc.gnn_encoder
    n, f = model.data["x"].shape[0], gcn.convs[0].lin.weight.shape[1]
    m = lambda seed, site, rows, cols, p: ops.dropout_mask(seed, site, rows, cols, p).double().cpu()   # noqa: E731
    return {
        "feat": m(enc.dropout_seed, ops.SITE_FEATURE, n, f, enc.feat_drop),
        "gcn": [m(gcn.dropout_seed, ops.SITE_GCN + i, n, c.lin.weight.shape[0], gcn.dropout) for i, c in enumerate(gcn.convs)],
        "att": [m(model.dropout_seed, ops.SITE_ATT + l, bs, model.num_heads * layer.att.out_channels, layer.dropout)
                for l, layer in enumerate(model.att_layers)],
        "score": m(score.dropout_seed, ops.SITE_MLP, bs, score.lins[0].weight.shape[0], score.dropout),
    }


def _ref_propagate(P, x, A, cfg, M):
    x = x * M["feat"]
    for i in range(cfg["gnn_layers"]):
        pre = f"node_encoder.gnn_encoder.convs.{i}"
        y = A @ (x @ P[f"{pre}.lin.weight"].t()) + P[f"{pre}.bias"]
        if cfg["layer_norm"]:
            ln = f"node_encoder.gnn_encoder.lns.{i}"
            y = F.layer_norm(y, y.shape[-1:], P[f"{ln}.weight"], P[f"{ln}.bias"], eps=1e-5)
        if cfg["relu"]:
            y = F.relu(y)
        y = y * M["gcn"][i]
        if cfg["residual"] and x.shape[-1] == y.shape[-1]:
            y = y + x
        x = y
    return F.layer_norm(x, x.shape[-1:], P["gnn_norm.weight"], P["gnn_norm.bias"], eps=1e-5)


def _ref_pairwise(links, X, sets, mode, P, cfg, att_masks):
    """oracle/ref_port.pairwise_features with each attention layer's output dropped by its mask."""
    bs, H = links.shape[1], cfg["num_heads"]
    order = [t for t in ("cn", "1hop", "non1hop") if t in sets]
    link_idx = torch.cat([sets[t][0][0] for t in order])
    node_idx = torch.cat([sets[t][0][1] for t in order])
    pes = []
    for t in order:
        _, pa, pb = sets[t]
        enc = ref_port._ENC[t]
        pes.append(ref_port._mlp(torch.stack((pa, pb)).t(), P, enc) + ref_port._mlp(torch.stack((pb, pa)).t(), P, enc))
    pe = torch.cat(pes, 0)
    feats = torch.cat((X[links[0]], X[links[1]]), -1)
    for l in range(cfg["trans_layers"]):
        pre = f"att_layers.{l}.att"
        x_i, x_j = feats[link_idx], X[node_idx]
        v = F.linear(torch.cat((x_j, pe), -1), P[f"{pre}.lin_r.weight"], P[f"{pre}.lin_r.bias"])
        C = v.shape[1] // H
        v = v.view(-1, H, C)
        e1, e2 = x_i.chunk(2, -1)
        e = (F.linear(e1, P[f"{pre}.lin_l.weight"], P[f"{pre}.lin_l.bias"]) +
             F.linear(e2, P[f"{pre}.lin_l.weight"], P[f"{pre}.lin_l.bias"])).view(-1, H, C)
        s = (F.leaky_relu(v * e, 0.2) * P[f"{pre}.att"]).sum(-1)
        alpha = ref_port._segment_softmax(s, link_idx, bs)
        msg = (v * alpha.unsqueeze(-1)).reshape(-1, H * C)
        out = torch.zeros((bs, H * C)).index_add_(0, link_idx, msg) + P[f"{pre}.bias"]
        feats = F.layer_norm(out, out.shape[-1:], P[f"att_layers.{l}.post_att_norm.weight"],
                             P[f"att_layers.{l}.post_att_norm.bias"]) * att_masks[l]

    def count(t):
        return torch.zeros(bs).index_add_(0, sets[t][0][0], torch.ones(sets[t][0].shape[1])).unsqueeze(-1)
    if mode == "cn":
        cols = [count("cn")]
    elif mode == "1-hop":
        cols = [count("cn"), count("1hop"), count("cn") + count("1hop")]
    else:
        cols = [count("cn"), count("1hop"), count("non1hop"), count("cn") + count("1hop")]
    return ref_port._mlp(torch.cat([feats] + cols, -1), P, "pairwise_lin")


def _ref_scores(P, Sp, x0, A, links, sets, mode, cfg, M):
    X = _ref_propagate(P, x0, A, cfg, M)
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        pw = _ref_pairwise(links, X, sets, mode, P, cfg, M["att"])
    finally:
        torch.set_default_dtype(old)
    el = ref_port._mlp(X[links[0]] * X[links[1]], P, "elementwise_lin")
    h = F.relu(F.linear(torch.cat((el, pw), -1), Sp["lins.0.weight"], Sp["lins.0.bias"])) * M["score"]
    return torch.sigmoid(F.linear(h, Sp["lins.1.weight"], Sp["lins.1.bias"])).squeeze(-1)


def _f64_params(module):
    return {k: v.detach().double().cpu().requires_grad_(True) for k, v in module.named_parameters()}


def _train_step(model, score, links, seed, adj_prop=None, adj_mask=None):
    """One seeded step (model -> score -> weighted loss -> backward); returns (prob, the CUDA generator state right
    before calc_pairwise: compute_node_mask from there keeps the pairs calc_pairwise kept)."""
    states = []
    real = model.calc_pairwise

    def spy(*args, **kwargs):
        states.append(torch.cuda.get_rng_state(DEV))
        return real(*args, **kwargs)
    model.calc_pairwise = spy
    try:
        for p in list(model.parameters()) + list(score.parameters()) + ([model.data["emb"].weight] if "emb" in model.data else []):
            p.grad = None
        torch.manual_seed(seed)
        w = torch.linspace(-1.0, 1.5, links.shape[1], device=DEV)
        prob = score(model(links, adj_prop=adj_prop, adj_mask=adj_mask))
        (prob * w).sum().backward()
    finally:
        del model.calc_pairwise
    return prob, states[0]


def _sets_after(model, links, state, adj_mask=None):
    torch.cuda.set_rng_state(state, DEV)
    infos = model.compute_node_mask(links, False, adj_mask)
    return {t: (info[0].cpu(), info[1].double().cpu(), info[2].double().cpu())
            for t, info in zip(("cn", "1hop", "non1hop"), infos) if info is not None}


def _clear_gcn_kinks(model, x0, A, M, margin=1e-5):
    """As in test_gpu_autograd: GCN biases shifted (seeded, 1e-3) until no ReLU input of the float64 propagate (with
    the masks) lies within `margin` of 0, where fp32 and float64 may take different sides of the kink."""
    cfg = model.train_args
    if not cfg["relu"]:
        return
    gen = torch.Generator().manual_seed(0)
    enc = model.node_encoder.gnn_encoder
    for _ in range(10):
        x, clear = x0 * M["feat"], True
        for i, conv in enumerate(enc.convs):
            y = A @ (x @ conv.lin.weight.detach().double().cpu().t()) + conv.bias.detach().double().cpu()
            if cfg["layer_norm"]:
                ln = enc.lns[i]
                y = F.layer_norm(y, y.shape[-1:], ln.weight.detach().double().cpu(), ln.bias.detach().double().cpu())
            if float(y.abs().min()) < margin:
                clear = False
                with torch.no_grad():
                    conv.bias.add_(1e-3 * torch.randn(conv.bias.shape, generator=gen, dtype=torch.float64).float().to(DEV))
                break
            y = F.relu(y) * M["gcn"][i]
            x = y + x if cfg["residual"] and x.shape[-1] == y.shape[-1] else y
        if clear:
            return
    raise AssertionError("could not move the GCN's ReLU inputs away from 0")


def _check_vs_float64(name, adj=False, seed=123):
    g = Golden(name)
    model, score = _build(g, **DROPS)
    model.train()
    score.train()
    links = torch.from_numpy(g["links"]).to(DEV)
    am = adj_prop = None
    if adj:
        am = g.masked_adjacency_coo(DEV)
        adj_prop = am.float()
    A = _dense_ahat(model, adj_prop)
    x0 = torch.from_numpy(g.features()).double()
    _train_step(model, score, links, seed, adj_prop, am)
    _clear_gcn_kinks(model, x0, A, _masks(model, score, links.shape[1]))      # (masks depend on the seed only)
    prob, state = _train_step(model, score, links, seed, adj_prop, am)
    M = _masks(model, score, links.shape[1])
    sets = _sets_after(model, links, state, am)
    S = sum(v[0].shape[1] for v in sets.values())
    assert S > 0
    P, Sp = _f64_params(model), _f64_params(score)
    E = None
    if "emb" in model.data:
        E = model.data["emb"].weight.detach().double().cpu().requires_grad_(True)
        x0 = E[model.data["x"].cpu().long()]
    ref = _ref_scores(P, Sp, x0, A, links.cpu(), sets, model.mask, dict(model.train_args), M)
    np.testing.assert_allclose(prob.detach().cpu().numpy(), ref.detach().numpy(), rtol=1e-5, atol=1e-5)
    (ref * torch.linspace(-1.0, 1.5, links.shape[1], dtype=torch.float64)).sum().backward()
    none_ref = {k for k, v in P.items() if v.grad is None}
    none_got = {k for k, v in model.named_parameters() if v.grad is None}
    assert none_got == none_ref, (none_got, none_ref)
    for k, p in model.named_parameters():
        if k not in none_ref:
            _close(p.grad, P[k].grad, k)
    for k, p in score.named_parameters():
        _close(p.grad, Sp[k].grad, "score." + k)
    if E is not None:
        _close(model.data["emb"].weight.grad, E.grad, "emb.weight")
    return model, sets


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_gradients_with_every_dropout_vs_float64(name):
    _check_vs_float64(name)


def test_node_dropout_on_a_merged_selection_vs_float64():
    """adj_prop / adj_mask supplied: node dropout runs on the merged (caller CN / 1-hop + stored >1-hop) selection."""
    _check_vs_float64("testset_d32", adj=True)


# ------------------------------------------------------------------------------------------------------- semantics
def test_eval_mode_ignores_dropout():
    g = Golden("all_d32")
    model, score = _build(g)
    dmodel, dscore = _build(g, **DROPS)
    links = torch.from_numpy(g["links"]).to(DEV)
    for m in (model, score, dmodel, dscore):
        m.eval()
    assert torch.equal(dscore(dmodel(links)), score(model(links)))
    X = dmodel.propagate()
    assert torch.equal(X, model.propagate())
    assert torch.equal(dmodel.calc_pairwise(links, X)[0], model.calc_pairwise(links, X)[0])


def test_no_grad_training_applies_dropout_detached():
    g = Golden("two_layers")
    model, score = _build(g, **DROPS)
    links = torch.from_numpy(g["links"]).to(DEV)
    model.eval()
    score.eval()
    ev = score(model(links))
    model.train()
    score.train()
    torch.manual_seed(5)
    with torch.no_grad():
        ng = score(model(links))
    assert not ng.requires_grad
    assert not torch.equal(ng, ev)
    torch.manual_seed(5)
    tr = score(model(links))
    assert tr.requires_grad
    assert torch.equal(tr.detach(), ng)           # same seeds, same kernels


def _loss(pos, neg):
    return -torch.log(pos + 1e-6).mean() - torch.log(1 - neg + 1e-6).mean()


def test_same_seed_same_step_and_different_seeds_differ():
    g = Golden("all_lowth_h2")
    model, score = _build(g, **DROPS)
    model.train()
    score.train()
    pos = torch.from_numpy(g["links"]).to(DEV)
    neg = torch.randint(0, g.n, tuple(pos.shape), generator=torch.Generator().manual_seed(4)).to(DEV)
    params = list(model.parameters()) + list(score.parameters())

    def step(seed):
        for p in params:
            p.grad = None
        torch.manual_seed(seed)
        loss = _loss(score(model(pos)), score(model(neg)))
        loss.backward()
        return loss.detach(), [None if p.grad is None else p.grad.clone() for p in params]
    l1, g1 = step(9)
    l2, g2 = step(9)
    l3, _ = step(10)
    assert torch.equal(l1, l2)
    for a, b in zip(g1, g2):
        assert (a is None) == (b is None)
        if a is not None:
            _close(b, a, "grad")
    assert not torch.equal(l1, l3)


def test_twenty_adam_steps_with_dropout_lower_the_loss():
    g = Golden("onehop_d64")
    model, score = _build(g, **DROPS)
    pos = torch.from_numpy(g["links"]).to(DEV)
    neg = torch.randint(0, g.n, tuple(pos.shape), generator=torch.Generator().manual_seed(4)).to(DEV)
    opt = torch.optim.Adam(list(model.parameters()) + list(score.parameters()), lr=1e-3)
    model.train()
    score.train()
    torch.manual_seed(0)
    losses = []
    for _ in range(20):
        opt.zero_grad()
        loss = _loss(score(model(pos)), score(model(neg)))
        loss.backward()
        opt.step()
        losses.append(float(loss.detach()))
    assert np.mean(losses[-5:]) < np.mean(losses[:5]), losses


# ------------------------------------------------------------------------------------------------ live reference
@pytest.mark.skipif(not os.path.isdir(os.environ.get("LPFORMER_REFERENCE_SRC", "")),
                    reason="needs the original LPFormer sources (LPFORMER_REFERENCE_SRC)")
def test_gradients_vs_live_reference_with_our_masks():
    """The unmodified reference with its F.dropout calls and drop_pairwise replaced, in call order, by our masks and
    kept pairs: parameter gradients at 1e-3 (fp32 on both sides)."""
    import sys
    import lpformer_b200 as L
    from lpformer_b200 import ops
    from oracle import lpformer_oracle as O
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    saved = list(sys.path)
    sys.path[:0] = [os.path.join(repo, "oracle", "shims"), os.environ["LPFORMER_REFERENCE_SRC"]]
    try:
        import models.link_transformer as RLT
        import models.other_models as ROM
        import modules.layers as RL
        import modules.node_encoder as RNE
    finally:
        sys.path[:] = saved
    rng = np.random.default_rng(21)
    torch.manual_seed(21)
    n, m = 110, 500
    e = rng.integers(0, n, (2, m))
    e = e[:, e[0] != e[1]]
    e = np.unique(np.concatenate([e, e[::-1]], 1), axis=1)
    e = e[:, np.lexsort((e[1], e[0]))]
    indptr = np.zeros(n + 1, np.int64)
    np.add.at(indptr, e[0] + 1, 1)
    indptr = np.cumsum(indptr)
    ppr = O.ppr_push(indptr, e[1].astype(np.int64), 0.15, 2e-3)
    prow = np.repeat(np.arange(n), np.diff(ppr.indptr))
    ei = torch.from_numpy(e.astype(np.int64))
    adj_t = torch.sparse_coo_tensor(ei, torch.ones(ei.shape[1]), (n, n)).coalesce()
    ppr_t = torch.sparse_coo_tensor(torch.from_numpy(np.stack([prow, ppr.indices])), torch.from_numpy(ppr.val),
                                    (n, n)).coalesce()
    data = {"x": torch.randn(n, 9), "adj_t": adj_t, "adj_mask": adj_t.bool().int(), "ppr": ppr_t, "full_adj_t": adj_t,
            "full_adj_mask": adj_t.bool().int(), "ppr_test": ppr_t}
    targs = dict(dim=12, num_heads=1, trans_layers=2, gnn_layers=2, residual=True, layer_norm=True, relu=True,
                 thresh_cn=2e-3, thresh_1hop=2e-3, thresh_non1hop=5e-3, **DROPS)
    links = torch.from_numpy(np.concatenate([e[:, rng.integers(0, e.shape[1], 50)], rng.integers(0, n, (2, 60))],
                                            1).astype(np.int64))
    w = torch.linspace(-1.0, 1.5, links.shape[1])
    model = L.LinkTransformer(dict(targs), {k: v.to(DEV) for k, v in data.items()}, device=DEV).to(DEV).train()
    score = L.mlp_score(model.out_dim, model.out_dim, 1, 2, dropout=PRED_DROP).to(DEV).train()
    prob, state = _train_step(model, score, links.to(DEV), 31)
    M = _masks(model, score, links.shape[1])
    torch.cuda.set_rng_state(state, DEV)
    kept = [(i[0].cpu(), i[1].cpu(), i[2].cpu()) if i is not None else None
            for i in model.compute_node_mask(links.to(DEV), False, None)]
    # our masks, in the order the reference calls F.dropout: features, GCN layers, attention layers, score head
    queue = [M["feat"]] + M["gcn"] + M["att"] + [M["score"]]
    real_dropout = F.dropout

    def dropout(x, p=0.5, training=True, inplace=False):
        if not training or p == 0:
            return x
        return x * queue.pop(0).float()
    ref = RLT.LinkTransformer(dict(targs), data, device="cpu").train()
    rscore = ROM.mlp_score(ref.out_dim, ref.out_dim, 1, 2, dropout=PRED_DROP).train()
    ref.load_state_dict(model.state_dict())
    rscore.load_state_dict(score.state_dict())
    mods = (RLT, ROM, RL, RNE)

    real_cnm = RLT.LinkTransformer.compute_node_mask
    try:
        for mod in mods:
            if hasattr(mod, "F"):
                mod.F.dropout = dropout
        # the sets after node dropout (compute_node_mask -> drop_pairwise) are ours
        RLT.LinkTransformer.compute_node_mask = lambda self, *a, **k: tuple(kept)
        (rscore(ref(links)) * w).sum().backward()
    finally:
        F.dropout = real_dropout
        for mod in mods:
            if hasattr(mod, "F"):
                mod.F.dropout = real_dropout
        RLT.LinkTransformer.compute_node_mask = real_cnm
    assert not queue, f"{len(queue)} masks left unused"
    rp = dict(ref.named_parameters())
    for k, p in model.named_parameters():
        assert (p.grad is None) == (rp[k].grad is None), k
        if p.grad is not None:
            _close(p.grad, rp[k].grad, k, rtol=1e-3)
    for (k, p), rq in zip(score.named_parameters(), rscore.parameters()):
        _close(p.grad, rq.grad, "score." + k, rtol=1e-3)
