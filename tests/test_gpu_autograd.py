"""-m gpu: the training path (autograd through propagate, calc_pairwise, elementwise_lin and mlp_score at dropout 0)
against float64 autograd of oracle/ref_port.py plus a float64 restatement of propagate, and the backward kernels alone
against float64 torch autograd.  Pass criterion for every gradient tensor: max abs error <= 1e-4 x max abs of the
float64 gradient."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import ref_port
from oracle.golden import GOLDEN_CASES, Golden

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
GRAD_RTOL = 1e-4


def _close(got, ref, name, rtol=GRAD_RTOL):
    assert got is not None, f"{name}: no gradient"
    got = got.detach().double().cpu()
    ref = ref.detach().double().cpu()
    assert got.shape == ref.shape, (name, got.shape, ref.shape)
    scale = float(ref.abs().max())
    err = float((got - ref).abs().max())
    assert err <= rtol * scale + 1e-12, f"{name}: max abs err {err:.3g} vs max abs {scale:.3g}"


# ------------------------------------------------------------------------------------------------- kernels alone
@pytest.mark.parametrize("n", [32, 64, 128, 256, 260])
@pytest.mark.parametrize("relu,norm", [(True, True), (False, True), (True, False)])
def test_layernorm_act_backward_kernel(n, relu, norm):
    from lpformer_b200 import ops
    torch.manual_seed(n)
    rows = 1237
    x = torch.randn(rows, n, device=DEV)
    g = (1 + 0.3 * torch.randn(n, device=DEV)) if norm else None
    b = 0.2 * torch.randn(n, device=DEV) if norm else None
    dy = torch.randn(rows, n, device=DEV)
    dg, db = (torch.empty(n, device=DEV), torch.empty(n, device=DEV)) if norm else (None, None)
    dx = ops.layernorm_act_backward(x, g, b, dy, relu=relu, dweight=dg, dbias=db)
    xd = x.double().cpu().requires_grad_(True)
    gd = g.double().cpu().requires_grad_(True) if norm else None
    bd = b.double().cpu().requires_grad_(True) if norm else None
    y = F.layer_norm(xd, (n,), gd, bd, eps=1e-5) if norm else xd
    if relu:
        y = F.relu(y)
    y.backward(dy.double().cpu())
    _close(dx, xd.grad, "dx")
    if norm:
        _close(dg, gd.grad, "dgamma")
        _close(db, bd.grad, "dbeta")


@pytest.mark.parametrize("M", [1, 1000, 100003])
@pytest.mark.parametrize("N,K", [(1, 64), (32, 32), (64, 128), (256, 256), (260, 260), (128, 2)])
def test_gemm_wgrad_and_dgrad_kernels(M, N, K):
    from lpformer_b200 import ops
    torch.manual_seed(M + N + K)
    A = torch.randn(M, K, device=DEV)
    dY = torch.randn(M, N, device=DEV)
    W = torch.randn(N, K, device=DEV)
    dW = torch.empty(N, K, device=DEV)
    db = torch.empty(N, device=DEV)
    ops.gemm_wgrad(A, dY, dW=dW, db=db)
    Ad, dYd = A.double().cpu(), dY.double().cpu()
    _close(dW, dYd.t() @ Ad, "dW")
    _close(db, dYd.sum(0), "db")
    ops.gemm_wgrad(A, dY, dW=dW, db=db, accumulate=True)
    _close(dW, 2 * dYd.t() @ Ad, "dW accumulated")
    _close(ops.linear_dgrad(dY, W), dYd @ W.double().cpu(), "dX")


def _attention_f64(ptr, node, KV, R, r_map, r_const, Q, att, bias, ln_w, ln_b, H, C, bs):
    """The attention of one layer in float64 autograd (modules/layers.py:161-224 in the algebra of attend.cu)."""
    cnt = (ptr[1:] - ptr[:-1]).view(3, bs)
    S = node.numel()
    link = torch.repeat_interleave(torch.arange(bs).repeat(3), (ptr[1:] - ptr[:-1]))
    rows = R[r_map.clamp(min=0)] if r_map is not None else R
    if r_map is not None:
        t = torch.repeat_interleave(torch.arange(3), torch.tensor([int(cnt[i].sum()) for i in range(3)]))
        rows = torch.where((r_map >= 0).unsqueeze(1), rows, r_const[t])
    v = (KV[node] + rows).view(S, H, C)
    q = Q[link].view(S, H, C)
    s = (F.leaky_relu(v * q, 0.2) * att.view(1, H, C)).sum(-1)
    idx = link.view(-1, 1).expand_as(s)                  # PyG softmax (SURVEY App. C), in float64
    mx = torch.full((bs, H), float("-inf"), dtype=torch.float64).scatter_reduce(0, idx, s, "amax", include_self=True)
    e = (s - mx[link]).exp()
    alpha = e / (torch.zeros((bs, H), dtype=torch.float64).scatter_add_(0, idx, e) + 1e-16)[link]
    out = torch.zeros((bs, H * C), dtype=torch.float64).index_add_(0, link, (v * alpha.unsqueeze(-1)).reshape(S, H * C))
    return F.layer_norm(out + bias, (H * C,), ln_w, ln_b, eps=1e-5)


@pytest.mark.parametrize("H,C", [(1, 32), (2, 32), (1, 64), (4, 16), (1, 128), (1, 256)])
@pytest.mark.parametrize("use_map", [False, True])
def test_attend_backward_kernel_large_links_and_row_map(H, C, use_map):
    """Links of 0, 1, 300 (> 256: the CTA-wide walk of the forward) and 3,000 pairs (> 1,024: the grid-wide split),
    with and without the (0, 0) row map (the shared row's gradient is the sum over its pairs)."""
    from lpformer_b200 import ops
    torch.manual_seed(H * C + use_map)
    N, HC = 5000, H * C
    sizes = [0, 1, 3000, 7, 300, 0, 40, 2]
    bs = len(sizes)
    per_type = [[int(s * f) for s in sizes] for f in (0.5, 0.3)]
    per_type.append([s - a - b for s, a, b in zip(sizes, *per_type)])
    counts = torch.tensor(sum(per_type, []), dtype=torch.int64)
    ptr = torch.zeros(3 * bs + 1, dtype=torch.int64)
    ptr[1:] = torch.cumsum(counts, 0)
    S = int(ptr[-1])
    node = torch.randint(0, N, (S,), dtype=torch.int32)
    KV = 0.5 * torch.randn(N, HC)
    Q = 0.5 * torch.randn(bs, HC)
    att = torch.randn(1, H, C) / C ** 0.5
    bias, ln_w, ln_b = 0.1 * torch.randn(HC), 1 + 0.2 * torch.randn(HC), 0.1 * torch.randn(HC)
    r_map = r_const = None
    if use_map:
        live = torch.rand(S) < 0.3
        t_of = torch.repeat_interleave(torch.arange(3), torch.tensor([int(sum(per_type[t])) for t in range(3)]))
        r_map = (torch.cumsum(live, 0) - 1).to(torch.int32)
        r_map = torch.where(live, r_map, (-1 - t_of).to(torch.int32))
        R = 0.5 * torch.randn(int(live.sum()), HC)
        r_const = 0.5 * torch.randn(3, HC)
    else:
        R = 0.5 * torch.randn(S, HC)
    dY = torch.randn(bs, HC)
    sel = ops.Selection("all", bs, ptr.to(DEV), node.to(DEV), None, None, None, (0, 0, 0, S), None)
    dKV = torch.zeros(N, HC, device=DEV)
    dR = torch.empty(R.shape, device=DEV)
    dRc = torch.zeros(3, HC, device=DEV) if use_map else None
    c = lambda t: None if t is None else t.to(DEV).contiguous()   # noqa: E731
    dQ, rows = ops.attend_backward(sel, c(KV), c(R), c(Q), c(att), c(bias), c(ln_w), c(ln_b), H, C, c(dY), dKV,
                                   r_map=c(r_map), r_const=c(r_const), dR=dR, dR_const=dRc)
    leaves = [t.double().requires_grad_(True) if t is not None else None
              for t in (KV, R, r_const, Q, att, bias, ln_w, ln_b)]
    y = _attention_f64(ptr, node.long(), leaves[0], leaves[1], None if r_map is None else r_map.long(), leaves[2],
                       *leaves[3:], H, C, bs)
    y.backward(dY.double())
    _close(dKV, leaves[0].grad, "dKV")
    _close(dR, leaves[1].grad, "dR")
    if use_map:
        _close(dRc, leaves[2].grad, "dR_const")
    _close(dQ, leaves[3].grad, "dQ")
    cs = torch.empty(4 * HC, device=DEV)
    ops.gemm_wgrad(None, rows, db=cs)
    _close(cs[3 * HC:].view(1, H, C), leaves[4].grad, "datt")
    _close(cs[:HC], leaves[5].grad, "dbias")
    _close(cs[HC:2 * HC], leaves[6].grad, "dln_w")
    _close(cs[2 * HC:3 * HC], leaves[7].grad, "dln_b")


@pytest.mark.parametrize("d", [32, 64, 128, 256])
def test_rpe_hidden_backward_kernel(d):
    from lpformer_b200 import ops
    torch.manual_seed(d)
    S = 20011
    pa, pb = torch.rand(S) * 0.5, torch.rand(S) * 0.5
    w1, b1 = torch.randn(d, 2), 0.1 * torch.randn(d)
    g, be = 1 + 0.2 * torch.randn(d), 0.1 * torch.randn(d)
    dh = torch.randn(S, d)
    grads = [torch.empty(d, 2, device=DEV)] + [torch.empty(d, device=DEV) for _ in range(3)]
    c = lambda t: t.to(DEV).contiguous()   # noqa: E731
    ops.rpe_hidden_backward(c(pa), c(pb), 0, S, c(w1), c(b1), c(g), c(be), c(dh), grads, False)
    L = [t.double().requires_grad_(True) for t in (w1, b1, g, be)]

    def h(x):
        return F.relu(F.layer_norm(F.linear(x, L[0], L[1]), (d,), L[2], L[3], eps=1e-5))
    xa = torch.stack((pa, pb), 1).double()
    (h(xa) + h(xa.flip(1))).backward(dh.double())
    for got, ref, name in zip(grads, L, ("w1", "b1", "ln_w", "ln_b")):
        _close(got, ref.grad, name)


# ------------------------------------------------------------------------------------------ whole model vs float64
def _build(g, emb_grad=False):
    import lpformer_b200 as L
    data = g.data_dict(DEV)
    if emb_grad and "emb" in data:
        data["emb"].weight.requires_grad_(True)
    model = L.LinkTransformer(g.train_args(), data, device=DEV).to(DEV)
    score = L.mlp_score(model.out_dim, model.out_dim, 1, 2).to(DEV)
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


def _ref_propagate(P, x, A, cfg):
    """propagate (reference models/link_transformer.py:110-129 with GCN models/other_models.py:61-76) in float64."""
    L = cfg["gnn_layers"]
    for i in range(L):
        pre = f"node_encoder.gnn_encoder.convs.{i}"
        xw = x @ P[f"{pre}.lin.weight"].t()
        y = A @ xw + P[f"{pre}.bias"]
        if cfg["layer_norm"]:
            ln = f"node_encoder.gnn_encoder.lns.{i}"
            y = F.layer_norm(y, y.shape[-1:], P[f"{ln}.weight"], P[f"{ln}.bias"], eps=1e-5)
        if cfg["relu"]:
            y = F.relu(y)
        if cfg["residual"] and x.shape[-1] == y.shape[-1]:
            y = y + x
        x = y
    return F.layer_norm(x, x.shape[-1:], P["gnn_norm.weight"], P["gnn_norm.bias"], eps=1e-5)


def _sets_of(model, links, adj_mask=None):
    infos = model.compute_node_mask(links, False, adj_mask)
    return {t: (info[0].cpu(), info[1].double().cpu(), info[2].double().cpu())
            for t, info in zip(("cn", "1hop", "non1hop"), infos) if info is not None}


def _ref_scores(P, Sp, x0, A, links, sets, mode, cfg):
    X = _ref_propagate(P, x0, A, cfg)
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        pw = ref_port.pairwise_features(links, X, sets, mode, P, cfg)
    finally:
        torch.set_default_dtype(old)
    el = ref_port._mlp(X[links[0]] * X[links[1]], P, "elementwise_lin")
    h = F.relu(F.linear(torch.cat((el, pw), -1), Sp["lins.0.weight"], Sp["lins.0.bias"]))
    return torch.sigmoid(F.linear(h, Sp["lins.1.weight"], Sp["lins.1.bias"])).squeeze(-1)


def _f64_params(module):
    return {k: v.detach().double().cpu().requires_grad_(True) for k, v in module.named_parameters()}


def _grad_check(model, score, links, x0_ref, A, sets, adj_prop=None, adj_mask=None):
    model.train()
    score.train()
    for p in list(model.parameters()) + list(score.parameters()):
        p.grad = None
    w = torch.linspace(-1.0, 1.5, links.shape[1], device=DEV)
    prob = score(model(links, adj_prop=adj_prop, adj_mask=adj_mask))
    (prob * w).sum().backward()
    P, Sp = _f64_params(model), _f64_params(score)
    cfg = dict(model.train_args)
    ref = _ref_scores(P, Sp, x0_ref, A, links.cpu(), sets, model.mask, cfg)
    np.testing.assert_allclose(prob.detach().cpu().numpy(), ref.detach().numpy(), rtol=1e-4, atol=1e-6)
    (ref * w.double().cpu()).sum().backward()
    none_ref = {k for k, v in P.items() if v.grad is None}
    none_got = {k for k, v in model.named_parameters() if v.grad is None}
    assert none_got == none_ref, (none_got, none_ref)
    assert "node_encoder.feat_transform.weight" in none_got
    for k, p in model.named_parameters():
        if k not in none_ref:
            _close(p.grad, P[k].grad, k)
    for k, p in score.named_parameters():
        _close(p.grad, Sp[k].grad, "score." + k)
    return prob


def _clear_gcn_kinks(model, x0, A, margin=1e-5):
    """Shifts GCN biases (seeded, 1e-3) until no ReLU input of propagate lies within `margin` of 0 in float64: there
    fp32 and float64 may take different sides of the kink (onehop_d64 has one at 2.4e-8; plain fp32 torch autograd is
    then 2.6 % off in that layer's bias gradient), which is conditioning, not the kernels."""
    cfg = model.train_args
    if not cfg["relu"]:
        return
    gen = torch.Generator().manual_seed(0)
    enc = model.node_encoder.gnn_encoder
    for _ in range(10):
        x, clear = x0, True
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
            y = F.relu(y)
            x = y + x if cfg["residual"] and x.shape[-1] == y.shape[-1] else y
        if clear:
            return
    raise AssertionError("could not move the GCN's ReLU inputs away from 0")


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_gradients_of_every_parameter_vs_float64(name):
    """modes all / 1-hop / cn, H = 2, two attention layers, GCN with and without LN / ReLU / residual, thresh_cn > 0,
    emb input: every parameter's gradient against float64 autograd of ref_port + the float64 propagate."""
    g = Golden(name)
    model, score = _build(g)
    links = torch.from_numpy(g["links"]).to(DEV)
    sets = _sets_of(model, links)
    x0 = torch.from_numpy(g.features()).double()
    A = _dense_ahat(model)
    _clear_gcn_kinks(model, x0, A)
    _grad_check(model, score, links, x0, A, sets)


def test_gradient_reaches_the_embedding_module():
    g = Golden("emb_d16")
    model, score = _build(g, emb_grad=True)
    emb = model.data["emb"]
    links = torch.from_numpy(g["links"]).to(DEV)
    sets = _sets_of(model, links)
    model.train()
    score.train()
    w = torch.linspace(-1.0, 1.5, links.shape[1], device=DEV)
    (score(model(links)) * w).sum().backward()
    P, Sp = _f64_params(model), _f64_params(score)
    E = emb.weight.detach().double().cpu().requires_grad_(True)
    x0 = E[model.data["x"].cpu().long()]
    ref = _ref_scores(P, Sp, x0, _dense_ahat(model), links.cpu(), sets, model.mask, dict(model.train_args))
    (ref * w.double().cpu()).sum().backward()
    _close(emb.weight.grad, E.grad, "emb.weight")


def test_caller_supplied_adj_prop_and_adj_mask():
    """The reference's training loop passes adj_prop = the train graph without the batch's positives and adj_mask:
    converted per call, CN / 1-hop from the supplied table, gradients as float64."""
    g = Golden("testset_d32")
    model, score = _build(g)
    links = torch.from_numpy(g["links"]).to(DEV)
    am = g.masked_adjacency_coo(DEV)
    adj_prop = am.float()
    sets = _sets_of(model, links, am)
    x0 = torch.from_numpy(g.features()).double()
    _grad_check(model, score, links, x0, _dense_ahat(model, adj_prop), sets, adj_prop=adj_prop, adj_mask=am)


@pytest.mark.parametrize("name", ["all_d32", "two_layers", "cn_thresh"])
def test_training_forward_bit_identical_to_eval_and_gate(name):
    g = Golden(name)
    model, score = _build(g)
    links = torch.from_numpy(g["links"]).to(DEV)
    model.eval()
    score.eval()
    ev = score(model(links))
    assert not ev.requires_grad
    X_ev = model.propagate()
    pw_ev, _ = model.calc_pairwise(links, X_ev)
    model.train()
    score.train()
    with torch.no_grad():
        ng = score(model(links))
    assert not ng.requires_grad
    tr = score(model(links))
    assert tr.requires_grad
    X_tr = model.propagate()
    pw_tr, _ = model.calc_pairwise(links, X_tr)
    assert X_tr.requires_grad and pw_tr.requires_grad
    assert torch.equal(tr.detach(), ev) and torch.equal(ng, ev)
    assert torch.equal(X_tr.detach(), X_ev) and torch.equal(pw_tr.detach(), pw_ev)
    # the inference-only entry points stay detached in training mode
    assert not model.score_links(links, X_tr, score).requires_grad


def _loss(pos, neg):
    """reference train/train_model.py: -log(pos + 1e-6).mean() - log(1 - neg + 1e-6).mean()."""
    return -torch.log(pos + 1e-6).mean() - torch.log(1 - neg + 1e-6).mean()


def test_twenty_sgd_steps_match_float64():
    g = Golden("all_d32")
    model, score = _build(g)
    n = g.n
    pos = torch.from_numpy(g["links"]).to(DEV)
    gen = torch.Generator().manual_seed(3)
    neg = torch.randint(0, n, tuple(pos.shape), generator=gen).to(DEV)
    sets_p, sets_n = _sets_of(model, pos), _sets_of(model, neg)
    P, Sp = _f64_params(model), _f64_params(score)
    A = _dense_ahat(model)
    x0 = torch.from_numpy(g.features()).double()
    cfg = dict(model.train_args)
    lr = 0.05
    opt = torch.optim.SGD(list(model.parameters()) + list(score.parameters()), lr=lr)
    model.train()
    score.train()
    for _ in range(20):
        opt.zero_grad()
        _loss(score(model(pos)), score(model(neg))).backward()
        opt.step()
        for v in list(P.values()) + list(Sp.values()):
            v.grad = None
        ref = _loss(_ref_scores(P, Sp, x0, A, pos.cpu(), sets_p, model.mask, cfg),
                    _ref_scores(P, Sp, x0, A, neg.cpu(), sets_n, model.mask, cfg))
        ref.backward()
        with torch.no_grad():
            for v in list(P.values()) + list(Sp.values()):
                if v.grad is not None:
                    v -= lr * v.grad
    for k, p in model.named_parameters():
        _close(p, P[k], k, rtol=1e-3)
    for k, p in score.named_parameters():
        _close(p, Sp[k], "score." + k, rtol=1e-3)
    # the derived caches picked the steps up: eval mode after training equals a fresh model with the same weights
    model.eval()
    score.eval()
    fresh, fscore = _build(g)
    fresh.load_state_dict(model.state_dict())
    fscore.load_state_dict(score.state_dict())
    X = model.propagate()
    assert torch.equal(model.score_links(pos, X, score), fresh.score_links(pos, fresh.propagate(), fscore))


def test_twenty_adam_steps_lower_the_loss():
    g = Golden("onehop_d64")
    model, score = _build(g)
    pos = torch.from_numpy(g["links"]).to(DEV)
    neg = torch.randint(0, g.n, tuple(pos.shape), generator=torch.Generator().manual_seed(4)).to(DEV)
    opt = torch.optim.Adam(list(model.parameters()) + list(score.parameters()), lr=1e-3)
    model.train()
    score.train()
    losses = []
    for _ in range(20):
        opt.zero_grad()
        loss = _loss(score(model(pos)), score(model(neg)))
        loss.backward()
        for p in list(model.parameters()) + list(score.parameters()):
            assert p.grad is None or bool(torch.isfinite(p.grad).all())
        opt.step()
        losses.append(float(loss.detach()))
    assert losses[-1] < losses[0], losses


def _thinned_ppr(data, keep_mod):
    """The PPR tables with a deterministic share of their entries kept: pairs without an entry get PPR values (0, 0)."""
    for key in ("ppr", "ppr_test"):
        p = data[key].coalesce()
        ix, v = p.indices(), p.values()
        k = ((ix[0] * 7 + ix[1]) % keep_mod) == 0
        data[key] = torch.sparse_coo_tensor(ix[:, k], v[k], p.shape).coalesce()


@pytest.mark.parametrize("name,keep_mod", [("onehop_d64", 3), ("all_d32", 3), ("zero_1hop", 5), ("two_layers", 10)])
def test_gradients_with_the_zero_ppr_row_map(name, keep_mod):
    """With most selected pairs at PPR (0, 0) (thinned PPR tables, thresh_cn = 0) the forward reads one shared RPE row
    per type through the row map; its gradient is the sum over those pairs and reaches the encoders' first Linear /
    LayerNorm at (0, 0), W2 / b2 and lin_r through the folded products.  Checked: the map is in use, and every
    parameter's gradient against float64."""
    import lpformer_b200 as L
    g = Golden(name)
    data = g.data_dict(DEV)
    _thinned_ppr(data, keep_mod)
    model = L.LinkTransformer(g.train_args(), data, device=DEV).to(DEV)
    score = L.mlp_score(model.out_dim, model.out_dim, 1, 2).to(DEV)
    msd, ssd = g.state_dicts(DEV)
    model.load_state_dict(msd)
    score.load_state_dict(ssd)
    model.rpe_map_min_pairs = 1
    saved = []
    stack = model._attention_stack

    def spy(*args, **kwargs):
        res = stack(*args, **kwargs)
        saved.append(res[2])
        return res
    model._attention_stack = spy
    links = torch.from_numpy(g["links"]).to(DEV)
    sets = _sets_of(model, links)
    S = sum(v[0].shape[1] for v in sets.values())
    zero = sum(int(((v[1] == 0) & (v[2] == 0)).sum()) for v in sets.values())
    assert 2 * zero > S and zero < S, (zero, S)          # the map is taken, with live rows as well
    x0 = torch.from_numpy(g.features()).double()
    A = _dense_ahat(model)
    _clear_gcn_kinks(model, x0, A)
    _grad_check(model, score, links, x0, A, sets)
    assert any(st is not None and st["r_map"] is not None for st in saved)


# ------------------------------------------------------------------------------------ the small kernels alone
@pytest.mark.parametrize("d", [32, 64, 128, 256, 33])
def test_gather_links_backward_kernel(d):
    from lpformer_b200 import ops
    torch.manual_seed(d)
    N, bs = 3001, 20011
    X = torch.randn(N, d, device=DEV)
    links = torch.randint(0, N, (2, bs), device=DEV)
    links[:, :50] = 7                                         # repeated and self links
    idx = torch.randperm(bs, device=DEV)[:9999].to(torch.int32)
    ds, dp = torch.randn(9999, d, device=DEV), torch.randn(9999, d, device=DEV)
    dX = torch.zeros(N, d, device=DEV)
    ops.gather_links_backward(links, X, dX, dsum=ds, dprod=dp, idx=idx)
    Xd = X.double().cpu().requires_grad_(True)
    li = links.cpu()[:, idx.long().cpu()]
    ((Xd[li[0]] + Xd[li[1]]) * ds.double().cpu() + Xd[li[0]] * Xd[li[1]] * dp.double().cpu()).sum().backward()
    _close(dX, Xd.grad, "dX")


@pytest.mark.parametrize("rows,d", [(1, 32), (1237, 64), (100003, 260), (5000, 33)])
def test_scatter_rows_backward_kernel(rows, d):
    from lpformer_b200 import ops
    torch.manual_seed(rows + d)
    n = rows // 3
    idx = torch.randperm(rows, device=DEV)[:n].to(torch.int32)
    dG = torch.randn(rows, d, device=DEV)
    dsrc, dfill = ops.scatter_rows_backward(dG, idx)
    mask = torch.ones(rows, dtype=torch.bool)
    mask[idx.long().cpu()] = False
    G = dG.double().cpu()
    if n > 0:
        _close(dsrc, G[idx.long().cpu()], "dsrc")
    _close(dfill, G[mask].sum(0), "dfill")


@pytest.mark.parametrize("rows,n", [(1, 1), (1237, 64), (20011, 33)])
def test_act_backward_kernel(rows, n):
    from lpformer_b200 import ops
    from lpformer_b200._lib import EPI_RELU, EPI_SIGMOID
    torch.manual_seed(rows)
    z = torch.randn(rows, n, dtype=torch.float64)
    dy = torch.randn(rows, n, device=DEV)
    for act, f in ((EPI_RELU, torch.relu), (EPI_SIGMOID, torch.sigmoid)):
        zd = z.clone().requires_grad_(True)
        y = f(zd)
        y.backward(dy.double().cpu())
        _close(ops.act_backward(y.detach().float().to(DEV), dy, act), zd.grad, f"act {act}")


@pytest.mark.skipif(not __import__("os").path.isdir(__import__("os").environ.get("LPFORMER_REFERENCE_SRC", "")),
                    reason="needs the original LPFormer sources (LPFORMER_REFERENCE_SRC)")
@pytest.mark.parametrize("cfg", [
    dict(dim=8, num_heads=2, trans_layers=1, gnn_layers=1, residual=False, layer_norm=True, relu=False, thresh_cn=0,
         thresh_1hop=1e-3, thresh_non1hop=1),                                              # 1-hop mode, H = 2
    dict(dim=12, num_heads=1, trans_layers=2, gnn_layers=2, residual=True, layer_norm=True, relu=True,
         thresh_cn=2e-3, thresh_1hop=2e-3, thresh_non1hop=5e-3)])                          # mode all, two layers
def test_gradients_vs_live_reference(cfg):
    """The unmodified reference (imported through oracle/shims as tests/test_reference_live.py does) in training mode
    at dropout 0, on CPU in fp32: its loss.backward() against ours, parameter by parameter (fp32 on both sides, so
    1e-3 of the max gradient), with the same None-gradient set."""
    import os
    import sys
    import lpformer_b200 as L
    from oracle import lpformer_oracle as O
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    saved = list(sys.path)
    sys.path[:0] = [os.path.join(repo, "oracle", "shims"), os.environ["LPFORMER_REFERENCE_SRC"]]
    try:
        from models.link_transformer import LinkTransformer as RefLT
        from models.other_models import mlp_score as RefScore
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
    targs = dict(cfg, dropout=0, gnn_drop=0, feat_drop=0, att_drop=0)
    ref = RefLT(dict(targs), data, device="cpu").train()
    rscore = RefScore(ref.out_dim, ref.out_dim, 1, 2).train()
    with torch.no_grad():
        for k, p in list(ref.named_parameters()) + list(rscore.named_parameters()):
            if "norm" in k or "lns" in k or k.endswith("bias"):
                p.add_(0.1 * torch.randn_like(p))
    links = torch.from_numpy(np.concatenate([e[:, rng.integers(0, e.shape[1], 50)], rng.integers(0, n, (2, 60))],
                                            1).astype(np.int64))
    w = torch.linspace(-1.0, 1.5, links.shape[1])
    (rscore(ref(links)) * w).sum().backward()
    model = L.LinkTransformer(dict(targs), {k: v.to(DEV) for k, v in data.items()}, device=DEV).to(DEV).train()
    score = L.mlp_score(model.out_dim, model.out_dim, 1, 2).to(DEV).train()
    model.load_state_dict(ref.state_dict())
    score.load_state_dict(rscore.state_dict())
    (score(model(links.to(DEV))) * w.to(DEV)).sum().backward()
    rp = dict(ref.named_parameters())
    for k, p in model.named_parameters():
        assert (p.grad is None) == (rp[k].grad is None), k
        if p.grad is not None:
            _close(p.grad, rp[k].grad, k, rtol=1e-3)
    for (k, p), rq in zip(score.named_parameters(), rscore.parameters()):
        _close(p.grad, rq.grad, "score." + k, rtol=1e-3)
