"""autograd Functions of the training path: at dropout 0 every forward runs the same kernels as the inference path, so
the values are bit-identical to eval mode, and every backward runs the kernels of csrc/backward.cu.  With dropout the
forwards apply the masks of csrc/dropout.cu (seed and site per call) and the backwards regenerate them from the seed:
no mask is stored.  PyTorch does the plumbing only: allocation, weight-sized products (the gradients of the folded
weights mapped back onto the reference's parameters) and the autograd graph.

Used by lpformer_b200.model when a module is in training mode and grad mode is enabled."""
from __future__ import annotations

import torch

from . import ops
from ._lib import EPI_NONE, EPI_RELU, EPI_SIGMOID, require_cuda
from .ops import _rowmajor


def _zeros_like(p):
    return torch.zeros_like(p, memory_format=torch.contiguous_format)


# ---------------------------------------------------------------------------------------------------------------- MLP
class MLPFunction(torch.autograd.Function):
    """Linear -> [LayerNorm] -> ReLU [-> dropout] ... -> Linear [-> sigmoid] (MLP.forward / mlp_score.forward) over the
    rows of x.  params: (W_0, b_0, ..., W_L, b_L[, norm.weight, norm.bias]) — the LayerNorm is shared by every hidden
    layer.  p > 0: hidden layer i is dropped with the mask (seed, SITE_MLP + i), row = row of x."""

    @staticmethod
    def forward(ctx, x, norm, sigmoid, p, seed, *params):
        n_lin = (len(params) - (2 if norm else 0)) // 2
        lins = [(params[2 * i], params[2 * i + 1]) for i in range(n_lin)]
        g, b = (params[-2], params[-1]) if norm else (None, None)
        inputs, pre = [], []
        h = x
        for i, (W, bias) in enumerate(lins[:-1]):
            inputs.append(h)
            if norm:
                z = ops.linear(h, W, bias)
                pre.append(z)
                h = ops.layernorm_act(z, g, b, relu=True)
            else:
                h = ops.linear(h, W, bias, epilogue=EPI_RELU)
                pre.append(h)      # (dropped in place below: [h > 0] still selects the gradient, see backward)
            if p > 0:
                ops.dropout(h, p, seed, ops.SITE_MLP + i, out=h)   # the dropped rows feed the next layer and its dW
        inputs.append(h)
        W, bias = lins[-1]
        out = ops.linear(h, W, bias, epilogue=EPI_SIGMOID if sigmoid else EPI_NONE)
        ctx.norm, ctx.sigmoid, ctx.n_lin, ctx.p, ctx.seed = norm, sigmoid, n_lin, p, seed
        ctx.save_for_backward(out, *inputs, *pre, *params)
        return out

    @staticmethod
    def backward(ctx, dout):
        n = ctx.n_lin
        saved = ctx.saved_tensors
        out, inputs, pre, params = saved[0], saved[1:1 + n], saved[1 + n:2 * n], saved[2 * n:]
        g, b = (params[-2], params[-1]) if ctx.norm else (None, None)
        grads = [None] * len(params)
        dn = (_zeros_like(g), _zeros_like(b)) if ctx.norm else None
        dy = dout.float()
        if ctx.sigmoid:
            dy = ops.act_backward(out, dy, EPI_SIGMOID)
        dx = None
        for i in range(n - 1, -1, -1):
            W, bias = params[2 * i], params[2 * i + 1]
            dW = _zeros_like(W)
            db = _zeros_like(bias) if bias is not None else None
            ops.gemm_wgrad(inputs[i], dy, dW=dW, db=db)
            grads[2 * i], grads[2 * i + 1] = dW, db
            if i == 0 and not ctx.needs_input_grad[0]:
                break
            dh = ops.linear_dgrad(dy, W)
            if i > 0 and ctx.p > 0:
                # the mask zeroes dh where the ReLU / LayerNorm output was dropped, so their backward needs nothing else
                ops.dropout(dh, ctx.p, ctx.seed, ops.SITE_MLP + i - 1, out=dh)
            if i == 0:
                dx = dh
            elif ctx.norm:
                dy = ops.layernorm_act_backward(pre[i - 1], g, b, dh, relu=True, dweight=dn[0], dbias=dn[1],
                                                accumulate_param=True)
            else:
                dy = ops.act_backward(pre[i - 1], dh, EPI_RELU)
        if ctx.norm:
            grads[-2], grads[-1] = dn
        return (dx, None, None, None, None, *grads)


def mlp_params(lins, norm):
    ps = []
    for lin in lins:
        ps += [lin.weight, lin.bias]
    if norm is not None:
        ps += [norm.weight, norm.bias]
    return ps


# ---------------------------------------------------------------------------------------------------------- GCN layer
class GCNLayerFunction(torch.autograd.Function):
    """One GCN layer (GCN.forward, reference models/other_models.py:61-76): out = LN2(res + drop(act(LN(A_hat x W^T +
    b)))), where res = x when `residual`; LN / LN2 optional; drop = dropout (p, seed, site) or nothing when dropout is
    None.  adj_t: the transpose of adj (adj itself when symmetric)."""

    @staticmethod
    def forward(ctx, x, W, bias, ln_w, ln_b, ln2_w, ln2_b, adj, adj_t, relu, residual, dropout=None):
        xw = ops.linear(x, W)
        ln = None if ln_w is None else (ln_w, ln_b)
        ln2 = None if ln2_w is None else (ln2_w, ln2_b)
        out = ops.gcn_layer(adj, xw, bias, ln=ln, relu=relu, residual=x if residual else None, ln2=ln2, dropout=dropout)
        ctx.adj, ctx.adj_t, ctx.relu, ctx.residual, ctx.dropout = adj, adj_t, relu, residual, dropout
        ctx.has_ln, ctx.has_ln2 = ln is not None, ln2 is not None
        ctx.save_for_backward(x, xw, W, bias, ln_w, ln_b, ln2_w, ln2_b)
        return out

    @staticmethod
    def backward(ctx, dout):
        x, xw, W, bias, ln_w, ln_b, ln2_w, ln2_b = ctx.saved_tensors
        dout = dout.float()
        y = ops.gcn_spmm(ctx.adj, xw, bias)                     # pre-norm rows (recomputed)
        g_ln2 = g_ln2b = g_ln = g_lnb = None
        du = dout
        if ctx.has_ln2:
            if ctx.has_ln or ctx.relu or ctx.residual or ctx.dropout is not None:
                u = ops.layernorm_act(y, ln_w, ln_b, relu=ctx.relu, residual=x if ctx.residual else None,
                                      dropout=ctx.dropout)
            else:
                u = y
            g_ln2, g_ln2b = _zeros_like(ln2_w), _zeros_like(ln2_b)
            du = ops.layernorm_act_backward(u, ln2_w, ln2_b, dout, relu=False, dweight=g_ln2, dbias=g_ln2b)
        if ctx.has_ln:
            g_ln, g_lnb = _zeros_like(ln_w), _zeros_like(ln_b)
        dd = du if ctx.dropout is None else ops.dropout(_rowmajor(du), *ctx.dropout)     # (du may be autograd's dout)
        dy = ops.layernorm_act_backward(y, ln_w, ln_b, dd, relu=ctx.relu, dweight=g_ln, dbias=g_lnb)
        dxw = ops.gcn_spmm(ctx.adj_t, dy, None)
        dW, db = _zeros_like(W), _zeros_like(bias)
        ops.gemm_wgrad(x, dxw, dW=dW)
        ops.gemm_wgrad(None, dy, db=db)
        dx = None
        if ctx.needs_input_grad[0]:
            dx = ops.linear_dgrad(dxw, W)
            if ctx.residual:
                ops.layernorm_act_backward(du, None, None, du, relu=False, dx=dx, accumulate_dx=True)   # dx += du
        return dx, dW, db, g_ln, g_lnb, g_ln2, g_ln2b, None, None, None, None, None


class DropoutFunction(torch.autograd.Function):
    """x * mask / (1 - p) of (seed, site), row = row of x (the feature dropout in front of the first GCN layer).  The
    dropped rows are the output (the next layer saves them for its weight gradient); the backward regenerates the mask."""

    @staticmethod
    def forward(ctx, x, p, seed, site):
        ctx.drop = (p, seed, site)
        return ops.dropout(_rowmajor(x), p, seed, site)

    @staticmethod
    def backward(ctx, dout):
        return ops.dropout(_rowmajor(dout.float()), *ctx.drop), None, None, None


# ------------------------------------------------------------------------------------------------------- link gathers
class GatherLinksFunction(torch.autograd.Function):
    """X[a] * X[b] (prod=True) or X[a] + X[b] of every link, or of the batch positions in idx."""

    @staticmethod
    def forward(ctx, X, links, idx, prod):
        s, p = ops.gather_links(links, X, want_sum=not prod, want_prod=prod, idx=idx)
        ctx.prod = prod
        ctx.save_for_backward(X, links, idx)
        return p if prod else s

    @staticmethod
    def backward(ctx, dout):
        X, links, idx = ctx.saved_tensors
        dX = torch.zeros_like(X, memory_format=torch.contiguous_format)
        dout = dout.float()
        ops.gather_links_backward(links, X, dX, dsum=None if ctx.prod else dout, dprod=dout if ctx.prod else None, idx=idx)
        return dX, None, None, None


# -------------------------------------------------------------------------------------- empty-set rows / concatenation
class ScatterFillFunction(torch.autograd.Function):
    """[bs, d] rows: fill_row everywhere, rows[j] at batch position idx[j] (calc_pairwise's compaction of the links with
    empty node sets).  The fill row's gradient is the sum over the rows idx does not name: it goes through the chain
    that built the row once, not once per link."""

    @staticmethod
    def forward(ctx, rows, fill_row, idx, bs):
        out = torch.empty((bs, fill_row.shape[-1]), dtype=torch.float32, device=fill_row.device)
        ops.scatter_rows(rows, idx, out, fill_row=fill_row.reshape(-1).contiguous())
        ctx.save_for_backward(idx)
        ctx.rows_none = rows is None
        return out

    @staticmethod
    def backward(ctx, dout):
        (idx,) = ctx.saved_tensors
        dsrc, dfill = ops.scatter_rows_backward(dout.float(), idx, want_src=not ctx.rows_none)
        return dsrc, dfill.view(1, -1), None, None


class ConcatFunction(torch.autograd.Function):
    """[a | b] along the columns, written by the row-copy kernel (lpf_layernorm_act without a norm); the gradient
    halves are views."""

    @staticmethod
    def forward(ctx, a, b):
        out = torch.empty((a.shape[0], a.shape[1] + b.shape[1]), dtype=torch.float32, device=a.device)
        ops.layernorm_act(a, None, None, out=out[:, : a.shape[1]])
        ops.layernorm_act(b, None, None, out=out[:, a.shape[1]:])
        ctx.split = a.shape[1]
        return out

    @staticmethod
    def backward(ctx, dout):
        return dout[:, : ctx.split], dout[:, ctx.split:]


# ------------------------------------------------------------------------------------------- RPE + attention layers
def pairwise_params(model):
    """The parameters the attention stack reads, in PairwiseFunction's order: per attention layer (lin_l.weight,
    lin_l.bias, lin_r.weight, lin_r.bias, att, bias, post_att_norm.weight, post_att_norm.bias), then per PPR encoder
    (linears.0.weight, linears.0.bias, norm.weight, norm.bias, linears.1.weight, linears.1.bias)."""
    ps = []
    for layer in model.att_layers:
        a = layer.att
        ps += [a.lin_l.weight, a.lin_l.bias, a.lin_r.weight, a.lin_r.bias, a.att, a.bias, layer.post_att_norm.weight,
               layer.post_att_norm.bias]
    for enc in model._encoders():
        ps += [enc.linears[0].weight, enc.linears[0].bias, enc.norm.weight, enc.norm.bias, enc.linears[1].weight,
               enc.linears[1].bias]
    return ps


class PairwiseFunction(torch.autograd.Function):
    """RPE -> attention layers -> counts of calc_pairwise (reference models/link_transformer.py:132-178) for the batch
    positions in idx (all links when None), before pairwise_lin.  The selection is a constant (as in the reference:
    the counts carry no gradient).  Returns [n, H*C + count_dim] (and the per-pair attention weights when asked)."""

    @staticmethod
    def forward(ctx, X, model, batch, sel, idx, want_alpha, drop, *params):
        feats, alpha, st = model._attention_stack(batch, X, sel, idx, want_alpha=want_alpha, save=True, drop=drop)
        ctx.model, ctx.sel, ctx.st, ctx.n_params, ctx.drop = model, sel, st, len(params), drop
        ctx.save_for_backward(X, batch, idx)
        if alpha is not None:
            ctx.mark_non_differentiable(alpha)
            return feats, alpha
        return feats

    @staticmethod
    def backward(ctx, dfeats, dalpha=None):
        X, batch, idx = ctx.saved_tensors
        model, sel, st = ctx.model, ctx.sel, ctx.st
        d, H = model.dim, model.num_heads
        L = model.num_layers
        encs = model._encoders()
        grads = {}
        dev = X.device
        csel, r_map = st["csel"], st["r_map"]
        S = sel.total
        HCs = [H * layer.att.out_channels for layer in model.att_layers]
        off = [sum(HCs[:l]) for l in range(L)]
        tot = sum(HCs)
        Sc = csel.total
        dKV = torch.zeros((X.shape[0], tot), dtype=torch.float32, device=dev) if S > 0 else None
        dR = torch.empty((Sc, tot), dtype=torch.float32, device=dev) if Sc > 0 else None
        # the shared (0, 0) rows' gradients, per layer (lpf_attend_backward adds into a contiguous [3, H*C] table)
        dRc = [torch.zeros((3, hc), dtype=torch.float32, device=dev) for hc in HCs] if r_map is not None else None
        g = ops._rowmajor(dfeats.float()[:, : HCs[-1]])
        drop = ctx.drop
        dxsum = None
        for l in range(L - 1, -1, -1):
            layer = model.att_layers[l]
            if drop is not None and drop[0][l] > 0:     # layer l's output was dropped: the same mask on its gradient
                g = ops.dropout(g, drop[0][l], drop[1], ops.SITE_ATT + l, out=None if l == L - 1 else g)
            att = layer.att
            C, HC = att.out_channels, HCs[l]
            Q, R, r_const, feats_in = st["Q"][l], st["R"][l], st["r_const"][l], st["feats_in"][l]
            dKV_l = dKV[:, off[l]:off[l] + HC] if dKV is not None else torch.zeros((1, HC), device=dev)
            dQ, rows = ops.attend_backward(sel, st["kvs"][l], R, Q, att.att, att.bias, layer.post_att_norm.weight,
                                           layer.post_att_norm.bias, H, C, g, dKV_l, idx=idx, r_map=r_map, r_const=r_const,
                                           dR=None if dR is None else dR[:, off[l]:off[l] + HC],
                                           dR_const=None if dRc is None else dRc[l])
            cs = torch.empty(4 * HC, dtype=torch.float32, device=dev)
            ops.gemm_wgrad(None, rows, db=cs)
            grads[(l, "bias")], grads[(l, "ln_w")], grads[(l, "ln_b")] = cs[:HC], cs[HC:2 * HC], cs[2 * HC:3 * HC]
            grads[(l, "att")] = cs[3 * HC:].view(1, H, C)
            # Q = xsum W_l^T + 2 b_l (layer 0) or [e1 | e2] [W_l | W_l]^T + 2 b_l (layer 1)
            dWl, dbl = _zeros_like(att.lin_l.weight), _zeros_like(att.lin_l.bias)
            if l == 0:
                ops.gemm_wgrad(feats_in, dQ, dW=dWl, db=dbl)
                dxsum = ops.linear_dgrad(dQ, att.lin_l.weight) if ctx.needs_input_grad[0] else None
            else:
                half = feats_in.shape[1] // 2
                ops.gemm_wgrad(feats_in[:, :half], dQ, dW=dWl, db=dbl)
                ops.gemm_wgrad(feats_in[:, half:], dQ, dW=dWl, accumulate=True)
                g = ops.linear_dgrad(dQ, st["derived"][l]["w_l_cat"], cache=False)
            grads[(l, "lin_l.weight")], grads[(l, "lin_l.bias")] = dWl, dbl * 2.0
        # lin_r = [W_x | W_pe]: KV = X W_x^T  and  R = hsum (W_pe W2_t)^T + 2 W_pe b2_t + b_r per type
        hsum, h0 = st["hsum"], st["h0"]
        dWr = [_zeros_like(layer.att.lin_r.weight) for layer in model.att_layers]
        dbr = [_zeros_like(layer.att.lin_r.bias) for layer in model.att_layers]
        dX = None
        if dKV is not None:
            for l in range(L):
                ops.gemm_wgrad(X, dKV[:, off[l]:off[l] + HCs[l]], dW=dWr[l][:, :d])
            if ctx.needs_input_grad[0]:
                w_x = torch.cat([layer.att.lin_r.weight.detach()[:, :d] for layer in model.att_layers], 0)
                dX = ops.linear_dgrad(dKV, w_x, cache=False)
                ops.gather_links_backward(batch, X, dX, dsum=dxsum, idx=idx)
        dhsum = torch.empty((Sc, d), dtype=torch.float32, device=dev) if Sc > 0 else None
        dh0 = None
        enc_grads = []
        for t, enc in enumerate(encs):
            r0, r1 = csel.type_range(t)
            w2, b2 = enc.linears[1].weight.detach(), enc.linears[1].bias.detach()
            dW2, db2 = torch.zeros_like(w2), torch.zeros_like(b2)
            m_cat = torch.cat([st["derived"][l]["rpe"][t][0] for l in range(L)], 0)      # [sum HC, d]
            if r1 > r0:
                ops.linear_dgrad(dR[r0:r1], m_cat, out=dhsum[r0:r1], cache=False)
            if dRc is not None:       # (three rows: weight-sized)
                dh0_t = sum(dRc[l][t:t + 1] @ st["derived"][l]["rpe"][t][0] for l in range(L))
                dh0 = dh0_t if dh0 is None else torch.cat((dh0, dh0_t), 0)
            for l in range(L):
                HC = HCs[l]
                w_pe = model.att_layers[l].att.lin_r.weight.detach()[:, d:]
                dM, dc = torch.zeros((HC, d), device=dev), torch.zeros(HC, device=dev)
                if r1 > r0:
                    ops.gemm_wgrad(hsum[r0:r1], dR[r0:r1, off[l]:off[l] + HC], dW=dM, db=dc)
                if dRc is not None:
                    ops.gemm_wgrad(h0[t:t + 1], dRc[l][t:t + 1], dW=dM, db=dc, accumulate=True)
                # M = W_pe W2, c = 2 W_pe b2 + b_r (weight-sized products)
                dWr[l][:, d:] += dM @ w2.t() + 2.0 * torch.outer(dc, b2)
                dbr[l] += dc
                dW2 += w_pe.t() @ dM
                db2 += 2.0 * (w_pe.t() @ dc)
            g1 = [_zeros_like(enc.linears[0].weight), _zeros_like(enc.linears[0].bias), _zeros_like(enc.norm.weight),
                  _zeros_like(enc.norm.bias)]
            w1 = (enc.linears[0].weight, enc.linears[0].bias, enc.norm.weight, enc.norm.bias)
            ops.rpe_hidden_backward(csel.src_ppr, csel.tgt_ppr, r0, r1, *w1, dhsum[r0:r1] if r1 > r0 else None, g1, False)
            if dRc is not None:
                zeros = torch.zeros(3, device=dev)
                ops.rpe_hidden_backward(zeros, zeros, t, t + 1, *w1, dh0[t:t + 1], g1, True)
            enc_grads.append(g1 + [dW2, db2])
        out = []
        for l in range(L):
            out += [grads[(l, "lin_l.weight")], grads[(l, "lin_l.bias")], dWr[l], dbr[l], grads[(l, "att")],
                    grads[(l, "bias")], grads[(l, "ln_w")], grads[(l, "ln_b")]]
        for g1 in enc_grads:
            out += g1
        return (dX, None, None, None, None, None, None, *out)


def require_training_inputs(*tensors):
    """No CPU fallback in training mode either."""
    require_cuda(*tensors)
