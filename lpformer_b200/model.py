"""Host-side mirror of the reference's module surface for the pairwise-encoding path.

Same class names, constructor arguments, attributes, method signatures and state_dict keys
as the reference (models/link_transformer.py, models/other_models.py, modules/layers.py,
modules/node_encoder.py), so `from lpformer_b200 import LinkTransformer, mlp_score` drops
into src/train's eval loops (train/testing.py:14-121) and loads reference checkpoints
(util/utils.py:38-51) unchanged.  Every forward computation runs in the sm_100a kernels
behind include/lpformer_b200.h; there is no PyTorch or CPU fallback.

A module in training mode with grad mode enabled builds an autograd graph through the same kernels (autograd.py; the
backward kernels are in csrc/backward.cu), so the reference's training loop body runs.  In training mode every dropout
of the reference is applied on the device (csrc/dropout.cu): feat_drop, gnn_drop, the attention layers' dropout,
MLP / mlp_score dropout and node dropout (att_drop), with or without grad mode.  In eval mode or under torch.no_grad()
the outputs are detached, as before.  score_links / score_queries / LinkScoreStream and the plans are inference-only.
"""
from __future__ import annotations

import functools
import os

import math
from typing import Optional

import torch
import torch.nn as nn

from . import autograd as AG
from . import ops
from ._lib import EPI_NONE, EPI_RELU, EPI_SIGMOID, LpfError
from .graph import CSR, csr_from_sparse, gcn_normalise, transpose_csr


def _drop_p(module: nn.Module, p, *tensors) -> float:
    """The dropout probability a forward of `module` applies: p in training mode, 0 in eval mode (F.dropout semantics:
    p outside [0, 1] raises ValueError).  The masks exist on the device only: with p > 0 in training mode a CPU tensor
    raises NotImplementedError."""
    ops.check_p(p)
    if not module.training or p == 0:
        return 0.0
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise NotImplementedError("dropout runs on the device only (lpformer_b200 has no CPU path); got a "
                                      f"{t.device} tensor")
    return float(p)


def _seed(module: nn.Module, device):
    """Draws the module's dropout seed for this forward (kept as module.dropout_seed: the masks of the forward are
    ops.dropout_mask(module.dropout_seed, site, ...))."""
    module.dropout_seed = ops.draw_seed(device)
    return module.dropout_seed


def _differentiable(module: nn.Module) -> bool:
    """The training path runs when the module is in training mode and grad mode is enabled."""
    return module.training and torch.is_grad_enabled()


def _grad_if_training(fn):
    """Runs `fn` with grad mode as the caller has it when the module trains (see _differentiable), under no_grad
    otherwise (detached outputs, the inference path)."""
    @functools.wraps(fn)
    def wrapper(self, *args, **kwargs):
        if _differentiable(self):
            return fn(self, *args, **kwargs)
        with torch.no_grad():
            return fn(self, *args, **kwargs)
    return wrapper


class _GlorotLinear(nn.Module):
    """Parameter holder with PyG `Linear` semantics (torch_geometric.nn.dense.linear):
    weight [out,in] glorot-uniform, bias zeros."""

    def __init__(self, in_channels, out_channels, bias=True):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.weight = nn.Parameter(torch.empty(out_channels, in_channels))
        if bias:
            self.bias = nn.Parameter(torch.empty(out_channels))
        else:
            self.register_parameter("bias", None)
        self.reset_parameters()

    def reset_parameters(self):
        stdv = math.sqrt(6.0 / (self.weight.size(-2) + self.weight.size(-1)))
        with torch.no_grad():       # (in place on the Parameter itself: bumps _version, which keys the derived caches)
            self.weight.uniform_(-stdv, stdv)
            if self.bias is not None:
                self.bias.fill_(0)

    def forward(self, x):
        return ops.linear(x, self.weight, self.bias)


class MLP(nn.Module):
    """reference models/other_models.py:80-138: Linear -> LayerNorm -> ReLU (-> dropout) ... -> Linear."""

    def __init__(self, num_layers, in_channels, hid_channels, out_channels, drop=0, norm="layer", sigmoid=False,
                 bias=True):
        super().__init__()
        self.dropout = drop
        self.sigmoid = sigmoid
        if norm == "batch":
            raise NotImplementedError("norm='batch' is never used on the LPFormer path")
        self.norm = nn.LayerNorm(hid_channels) if norm == "layer" else None
        self.linears = nn.ModuleList()
        if num_layers == 1:
            self.linears.append(nn.Linear(in_channels, out_channels, bias=bias))
        else:
            self.linears.append(nn.Linear(in_channels, hid_channels, bias=bias))
            for _ in range(num_layers - 2):
                self.linears.append(nn.Linear(hid_channels, hid_channels, bias=bias))
            self.linears.append(nn.Linear(hid_channels, out_channels, bias=bias))

    def reset_parameters(self):
        for lin in self.linears:
            lin.reset_parameters()
        if self.norm is not None:
            self.norm.reset_parameters()

    @_grad_if_training
    def forward(self, x, out=None):
        p = _drop_p(self, self.dropout, x)
        lead = x.shape[:-1]
        x = x.reshape(-1, x.shape[-1])
        if torch.is_grad_enabled() or p > 0:
            AG.require_training_inputs(x)
            seed = _seed(self, x.device) if p > 0 else None
            x = AG.MLPFunction.apply(x, self.norm is not None, self.sigmoid, p, seed,
                                     *AG.mlp_params(self.linears, self.norm))
            if out is not None:
                out.copy_(x)
            return x.reshape(*lead, x.shape[-1]).squeeze(-1)
        for lin in list(self.linears)[:-1]:
            if self.norm is not None:
                x = ops.linear(x, lin.weight, lin.bias)
                x = ops.layernorm_act(x, self.norm.weight, self.norm.bias, relu=True, out=x)
            else:
                x = ops.linear(x, lin.weight, lin.bias, epilogue=EPI_RELU)
        last = self.linears[-1]
        x = ops.linear(x, last.weight, last.bias, out=out, epilogue=EPI_SIGMOID if self.sigmoid else EPI_NONE)
        x = x.reshape(*lead, x.shape[-1])
        return x.squeeze(-1)


class mlp_score(nn.Module):
    """reference models/other_models.py:142-179: Linear/ReLU ... Linear -> sigmoid -> squeeze."""

    def __init__(self, in_channels, hidden_channels, out_channels, num_layers, dropout=0):
        super().__init__()
        self.lins = nn.ModuleList()
        if num_layers == 1:
            self.lins.append(nn.Linear(in_channels, out_channels))
        else:
            self.lins.append(nn.Linear(in_channels, hidden_channels))
            for _ in range(num_layers - 2):
                self.lins.append(nn.Linear(hidden_channels, hidden_channels))
            self.lins.append(nn.Linear(hidden_channels, out_channels))
        self.dropout = dropout

    def reset_parameters(self):
        for lin in self.lins:
            lin.reset_parameters()

    @_grad_if_training
    def forward(self, x, return_logits=False):
        p = _drop_p(self, self.dropout, x)
        x = x.reshape(-1, x.shape[-1])
        if torch.is_grad_enabled() or p > 0:
            AG.require_training_inputs(x)
            seed = _seed(self, x.device) if p > 0 else None
            return AG.MLPFunction.apply(x, False, not return_logits, p, seed,
                                        *AG.mlp_params(self.lins, None)).squeeze(-1)
        for lin in list(self.lins)[:-1]:
            x = ops.linear(x, lin.weight, lin.bias, epilogue=EPI_RELU)
        last = self.lins[-1]
        x = ops.linear(x, last.weight, last.bias, epilogue=EPI_NONE if return_logits else EPI_SIGMOID)
        return x.squeeze(-1)


class GCNConv(nn.Module):
    """Parameter layout of PyG 2.2.0 GCNConv (`lin.weight` [out,in] without bias, `bias` [out])."""

    def __init__(self, in_channels, out_channels, cached=False, normalize=True):
        super().__init__()
        if not normalize:
            raise NotImplementedError("GCNConv(normalize=False) is never used by the reference")
        self.cached = cached
        self.lin = _GlorotLinear(in_channels, out_channels, bias=False)
        self.bias = nn.Parameter(torch.empty(out_channels))
        self.reset_parameters()

    def reset_parameters(self):
        self.lin.reset_parameters()
        with torch.no_grad():
            self.bias.fill_(0)

    @torch.no_grad()
    def forward(self, x, adj_norm: CSR, out=None, row0=0, rows=None):
        """A_hat @ (x W^T) + bias on an already gcn-normalised CSR (rows [row0,row0+rows))."""
        xw = ops.linear(x, self.lin.weight)
        return ops.gcn_spmm(adj_norm, xw, self.bias, out=out, row0=row0, rows=rows)


class GCN(nn.Module):
    """reference models/other_models.py:10-76."""

    def __init__(self, in_channels, hidden_channels, out_channels, num_layers, dropout, residual=False, cached=False,
                 normalize=True, layer_norm=True, relu=True):
        super().__init__()
        self.relu = relu
        self.convs = nn.ModuleList()
        if num_layers == 1:
            hidden_channels = out_channels
        self.convs.append(GCNConv(in_channels, hidden_channels, cached=cached, normalize=normalize))
        if layer_norm:
            self.lns = nn.ModuleList()
            self.lns.append(nn.LayerNorm(hidden_channels))
        else:
            self.lns = None
        if num_layers > 1:
            for _ in range(num_layers - 2):
                self.convs.append(GCNConv(hidden_channels, hidden_channels, cached=cached, normalize=normalize))
                self.lns.append(nn.LayerNorm(hidden_channels))
            self.convs.append(GCNConv(hidden_channels, out_channels, cached=cached, normalize=normalize))
            if layer_norm:
                self.lns.append(nn.LayerNorm(hidden_channels))
        self.dropout = dropout
        self.residual = residual

    def reset_parameters(self):
        for conv in self.convs:
            conv.reset_parameters()

    @_grad_if_training
    def forward(self, x, adj_norm: CSR, final_norm=None):
        """reference :61-76.  Per layer one contraction (x W^T) and ONE launch for the rest (SpMM + bias + LayerNorm +
        ReLU + residual, ops.gcn_layer); final_norm = (weight, bias) of a LayerNorm applied to the last layer's output
        in the same launch (LinkTransformer.gnn_norm).  Dropout (training mode, p = self.dropout) of every layer's
        activated rows rides in the same launch: mask (seed, SITE_GCN + layer), row = node id."""
        p = _drop_p(self, self.dropout, x)
        seed = _seed(self, x.device) if p > 0 else None
        drop = (lambda i: (p, seed, ops.SITE_GCN + i) if p > 0 else None)   # noqa: E731
        last = len(self.convs) - 1
        if torch.is_grad_enabled():
            AG.require_training_inputs(x)
            adj_t = transpose_csr(adj_norm)
            for i, conv in enumerate(self.convs):
                ln = self.lns[i] if self.lns is not None else None
                ln2 = final_norm if i == last else None
                x = AG.GCNLayerFunction.apply(x, conv.lin.weight, conv.bias, None if ln is None else ln.weight,
                                              None if ln is None else ln.bias, None if ln2 is None else ln2[0],
                                              None if ln2 is None else ln2[1], adj_norm, adj_t, self.relu,
                                              bool(self.residual and x.shape[-1] == conv.lin.weight.shape[0]), drop(i))
            return x
        for i, conv in enumerate(self.convs):
            xw = ops.linear(x, conv.lin.weight)
            ln = self.lns[i] if self.lns is not None else None
            res = x if (self.residual and x.shape[-1] == xw.shape[-1]) else None
            x = ops.gcn_layer(adj_norm, xw, conv.bias, ln=None if ln is None else (ln.weight, ln.bias), relu=self.relu,
                              residual=res, ln2=final_norm if i == last else None, dropout=drop(i))
        return x


class NodeEncoder(nn.Module):
    """reference modules/node_encoder.py:8-44 (feat_transform is allocated but unused there too)."""

    def __init__(self, data, train_args, device="cuda"):
        super().__init__()
        self.device = device
        self.dim = train_args["dim"]
        init_dim = self.dim if "emb" in data else data["x"].size(1)
        self.feat_drop = train_args.get("feat_drop", 0)
        self.feat_transform = nn.Linear(init_dim, self.dim)
        self.gnn_encoder = GCN(init_dim, self.dim, self.dim, train_args["gnn_layers"], train_args.get("gnn_drop", 0),
                               cached=train_args.get("gcn_cache"), residual=train_args["residual"],
                               layer_norm=train_args["layer_norm"], relu=train_args["relu"])

    @_grad_if_training
    def forward(self, features, adj_norm: CSR, test_set=False, final_norm=None):
        """Feature dropout (training mode, p = feat_drop; mask (seed, SITE_FEATURE), row = node id) in front of the GCN.
        The dropped features are stored (the first GCN layer saves its input for its weight gradient): one extra
        [N, F] fp32 table while the graph lives."""
        p = _drop_p(self, self.feat_drop, features)
        if p > 0:
            seed = _seed(self, features.device)
            if torch.is_grad_enabled():
                features = AG.DropoutFunction.apply(features, p, seed, ops.SITE_FEATURE)
            else:
                features = ops.dropout(ops._rowmajor(features), p, seed, ops.SITE_FEATURE)
        return self.gnn_encoder(features, adj_norm, final_norm=final_norm)


class LinkAttention(nn.Module):
    """Parameters of the reference's GATv2-style LinkAttention (modules/layers.py:88-158)."""

    def __init__(self, in_channels, out_channels, train_args, concat=True, negative_slope=0.2, bias=True,
                 node_dim=None, **kwargs):
        super().__init__()
        if not concat or not bias or negative_slope != 0.2:
            raise NotImplementedError("only concat=True, bias=True, negative_slope=0.2 (what the reference builds)")
        self.in_channels, self.out_channels = in_channels, out_channels
        self.heads = train_args["num_heads"]
        self.concat = concat
        self.negative_slope = negative_slope
        self.dropout = train_args.get("att_drop", 0)  # stored, never applied (as in the reference)
        node_dim = in_channels * 2 if node_dim is None else node_dim * 2
        self.lin_l = _GlorotLinear(in_channels, self.heads * out_channels, bias=True)
        self.lin_r = _GlorotLinear(node_dim, self.heads * out_channels, bias=True)
        self.att = nn.Parameter(torch.empty(1, self.heads, out_channels))
        self.bias = nn.Parameter(torch.empty(self.heads * out_channels))
        self.reset_parameters()

    def reset_parameters(self):
        self.lin_l.reset_parameters()
        self.lin_r.reset_parameters()
        stdv = math.sqrt(6.0 / (self.att.size(-2) + self.att.size(-1)))
        with torch.no_grad():
            self.att.uniform_(-stdv, stdv)
            self.bias.fill_(0)


class LinkTransformerLayer(nn.Module):
    """reference modules/layers.py:17-82 (parameters: att.*, post_att_norm.*)."""

    def __init__(self, dim, train_args, concat=True, out_dim=None, node_dim=None):
        super().__init__()
        self.dropout = train_args.get("dropout", 0)
        out_dim = dim if out_dim is None else out_dim
        self.att = LinkAttention(dim, out_dim, train_args, concat=concat, node_dim=node_dim)
        self.post_att_norm = nn.LayerNorm(out_dim * train_args["num_heads"] if concat else out_dim)


class _Tables:
    """CSR tables of one graph variant (train graph or test_set=True variant)."""

    def __init__(self):
        self.adj_mask: Optional[CSR] = None
        self.ppr: Optional[CSR] = None
        self.adj_norm: Optional[CSR] = None


class LinkTransformer(nn.Module):
    """Drop-in for reference models/link_transformer.py:16-482 (inference).

    forward(batch, adj_prop=None, adj_mask=None, test_set=False, return_weights=False) -> [BS, 2*dim]
    propagate(adj=None, test_set=False) -> [N, dim]
    calc_pairwise(batch, X_node, test_set=False, adj_mask=None, return_weights=False) -> ([BS, dim], att_weights|None)
    compute_node_mask(batch, test_set, adj) -> reference-format tuples of the selected sets
    elementwise_lin / pairwise_lin / ppr_encoder_* -> MLP modules,  out_dim == 2*dim
    """

    def __init__(self, train_args, data, device="cuda"):
        super().__init__()
        self.train_args = train_args
        self.data = data
        self.device = device

        self.thresh_cn = train_args["thresh_cn"]
        self.thresh_1hop = train_args["thresh_1hop"]
        self.thresh_non1hop = train_args["thresh_non1hop"]
        if self.thresh_non1hop == 1 and self.thresh_1hop == 1:
            self.mask = "cn"
        elif self.thresh_non1hop == 1 and self.thresh_1hop < 1:
            self.mask = "1-hop"
        else:
            self.mask = "all"

        self.dim = train_args["dim"]
        self.att_drop = train_args.get("att_drop", 0)
        self.num_layers = train_args["trans_layers"]
        self.num_heads = train_args["num_heads"]
        self.num_nodes = data["x"].shape[0]
        self.out_dim = self.dim * 2
        if self.num_layers > 2:
            raise NotImplementedError("trans_layers > 2 is shape-inconsistent in the reference as well")
        if self.num_layers == 2 and self.num_heads != 1:
            raise NotImplementedError("trans_layers == 2 requires num_heads == 1 (reference chunk(2) semantics)")

        self.gnn_norm = nn.LayerNorm(self.dim)
        self.node_encoder = NodeEncoder(data, train_args, device=device)

        self.att_layers = nn.ModuleList()
        att_inner_dim = self.dim * 2 if self.num_layers > 1 else self.dim
        self.att_layers.append(LinkTransformerLayer(self.dim, train_args, out_dim=att_inner_dim))
        for _ in range(self.num_layers - 2):
            self.att_layers.append(LinkTransformerLayer(self.dim, train_args, node_dim=self.dim))
        if self.num_layers > 1:
            self.att_layers.append(LinkTransformerLayer(self.dim, train_args, out_dim=self.dim, node_dim=self.dim))

        self.elementwise_lin = MLP(2, self.dim, self.dim, self.dim)
        self.ppr_encoder_cn = MLP(2, 2, self.dim, self.dim)
        if self.mask == "cn":
            count_dim = 1
        elif self.mask == "1-hop":
            self.ppr_encoder_onehop = MLP(2, 2, self.dim, self.dim)
            count_dim = 3
        else:
            count_dim = 4
            self.ppr_encoder_onehop = MLP(2, 2, self.dim, self.dim)
            self.ppr_encoder_non1hop = MLP(2, 2, self.dim, self.dim)
        self.count_dim = count_dim
        pairwise_dim = self.dim * train_args["num_heads"] + count_dim
        self.pairwise_lin = MLP(2, pairwise_dim, pairwise_dim, self.dim)

        self.register_load_state_dict_post_hook(lambda module, incompatible: module.invalidate_weights())
        self._tables = {False: _Tables(), True: _Tables()}
        self._derived = None        # folded weights, keyed by parameter versions
        self._kv_cache = None       # per-layer KV tables, keyed by the X_node they were built from
        self._pw_const_cache = None  # pairwise vector of a link with empty sets, keyed by parameter versions
        self._head_cache = None     # operands of the fused heads kernel
        self._plans = {}            # sync-free execution plans of score_links, keyed by batch size / X_node
        self._plan_cap = {}
        self.use_plans = True       # one-pass selection + device-side sizes (plan.py)
        self.use_graphs = True      # ... replayed as a CUDA graph
        # non-empty links below this share of the batch take the one-warp-per-link path (LPF_NZ_FUSED_SHARE: tuning knob)
        # "bf16": the sync-free plans (score_links / LinkScoreStream at d = 64) read X and KV from bf16 copies — half the
        # gather bytes; products, contractions and accumulation as in fp32 mode (north star: 1e-2 in bf16)
        self.node_dtype = os.environ.get("LPF_NODE_DTYPE", "f32")
        self._tab16 = None
        self.nz_fused_share = float(os.environ.get("LPF_NZ_FUSED_SHARE", 1.0 / 16))
        self.nz_fused_max_links = int(os.environ.get("LPF_NZ_FUSED_MAX_LINKS", 8192))
        self.rpe_map_min_pairs = int(os.environ.get("LPF_RPE_MAP_MIN_PAIRS", 1 << 18))   # pairs per batch: (0, 0) pairs share an RPE row
        self.nz_pairs_tc_min = int(os.environ.get("LPF_NZ_PAIRS_TC_MIN", 150000))   # pairs per batch: RPE stage on the tensor cores

    # ------------------------------------------------------------------ graph tables
    def _dev(self):
        return self.gnn_norm.weight.device

    def _weights_key(self, other=None):
        """Versions of every parameter (cheap: the parameter list is walked once and kept), so that the derived /
        packed weights are rebuilt after load_state_dict, .to() or an in-place update."""
        pl = self.__dict__.get("_plist")
        if pl is None:
            pl = self.__dict__["_plist"] = list(self.parameters())
        key = tuple([p._version for p in pl]) + (pl[0].device,)
        if other is not None:
            ol = other.__dict__.get("_plist")
            if ol is None:
                ol = other.__dict__["_plist"] = list(other.parameters())
            key += tuple([p._version for p in ol]) + (id(other),)
        return key

    def _graph_key(self, test_set, mask):
        suffix = "mask" if mask else "t"
        return f"full_adj_{suffix}" if test_set else f"adj_{suffix}"

    def get_adj(self, test_set=False, mask=False):
        """reference :389-397 — returns the HBM-resident CSR built from data[...]."""
        tab = self._tables[bool(test_set)]
        if mask:
            if tab.adj_mask is None:
                tab.adj_mask = csr_from_sparse(self.data[self._graph_key(test_set, True)], self._dev(), mask=True)
            return tab.adj_mask
        if tab.adj_norm is None:
            tab.adj_norm = gcn_normalise(csr_from_sparse(self.data[self._graph_key(test_set, False)], self._dev()))
        return tab.adj_norm

    def get_ppr(self, test_set=False):
        """reference :399-406."""
        use_test = bool(test_set and "ppr_test" in self.data)
        tab = self._tables[use_test]
        if tab.ppr is None:
            tab.ppr = csr_from_sparse(self.data["ppr_test" if use_test else "ppr"], self._dev())
        return tab.ppr

    def get_degree(self, test_set=False):
        if test_set and "degree_test" in self.data:
            return self.data["degree_test"]
        return self.data["degree"]

    def invalidate_graph_tables(self):
        """Call after mutating the sparse tensors inside `data`."""
        self._tables = {False: _Tables(), True: _Tables()}

    def invalidate_weights(self):
        """Drops everything derived from the parameters (folded weights, packed tensor-core images, K/V tables, the
        empty-set pairwise constant, head operands, execution plans and their CUDA graphs).  The caches are keyed on
        Parameter._version, which writes through `.data` (reset_parameters, some optimisers) do not bump: call this
        after such an update.  load_state_dict and reset_parameters call it themselves."""
        self._derived = None
        self._kv_cache = None
        self._pw_const_cache = None
        self._head_cache = None
        self._plans = {}
        self.__dict__.pop("_plist", None)
        ops.drop_packed_weights()

    # ------------------------------------------------------------------ folded weights
    def _encoders(self):
        enc = [self.ppr_encoder_cn]
        if self.mask != "cn":
            enc.append(self.ppr_encoder_onehop)
        if self.mask == "all":
            enc.append(self.ppr_encoder_non1hop)
        return enc

    def _get_derived(self):
        """Per (layer, type): M = W_pe W2_t  [HC,d]  and  c = 2 W_pe b2_t + b_r  [HC]
        (SURVEY App. B: lin_r([x | pe]) = W_x x + W_pe (W2 (h1+h2) + 2 b2) + b_r)."""
        key = self._weights_key()
        if self._derived is not None and self._derived[0] == key:
            return self._derived[1]
        d = self.dim
        out = []
        for layer in self.att_layers:
            w_r = layer.att.lin_r.weight.detach().double()
            w_pe = w_r[:, d:]
            per_type = []
            for enc in self._encoders():
                w2 = enc.linears[1].weight.detach().double()
                b2 = enc.linears[1].bias.detach().double()
                m = (w_pe @ w2).float().contiguous()
                c = (2.0 * (w_pe @ b2) + layer.att.lin_r.bias.detach().double()).float().contiguous()
                per_type.append((m, c))
            # lin_l(e1) + lin_l(e2) = [e1 | e2] [W_l | W_l]^T + 2 b_l for the chunked inputs of layers > 0
            w_l = layer.att.lin_l.weight.detach()
            out.append({"rpe": per_type, "w_l_cat": torch.cat((w_l, w_l), dim=1).contiguous()})
        self._derived = (key, out)
        return out

    def _get_kv(self, X_node):
        """KV_l = X W_x,l^T  [N, HC_l] for every attention layer; rebuilt when X_node changes."""
        key = (X_node.data_ptr(), X_node._version, tuple(X_node.shape),
               tuple(layer.att.lin_r.weight._version for layer in self.att_layers))
        if self._kv_cache is not None and self._kv_cache[0] == key:
            return self._kv_cache[1]
        d = self.dim
        kvs = [ops.linear(X_node, layer.att.lin_r.weight[:, :d]) for layer in self.att_layers]
        self._kv_cache = (key, kvs, X_node.detach())   # keep X_node alive so the pointer key stays valid
        return kvs

    def _prime_kv(self, X_node, kvs):
        """Install externally built K/V tables for X_node (multi-GPU all-gather path)."""
        key = (X_node.data_ptr(), X_node._version, tuple(X_node.shape),
               tuple(layer.att.lin_r.weight._version for layer in self.att_layers))
        self._kv_cache = (key, kvs, X_node)

    # ------------------------------------------------------------------ reference API
    @_grad_if_training
    def forward(self, batch, adj_prop=None, adj_mask=None, test_set=False, return_weights=False):
        """reference :82-107."""
        batch = ops.links_tensor(batch, self._dev())
        X_node = self.propagate(adj_prop, test_set)
        if torch.is_grad_enabled():
            # both halves carry gradients: each is built by its own Function, then joined by the row-copy kernel
            xprod = AG.GatherLinksFunction.apply(self._check_x(X_node), batch, None, True)
            el = self.elementwise_lin(xprod)
            pw, att_weights = self.calc_pairwise(batch, X_node, test_set, adj_mask=adj_mask, return_weights=return_weights)
            feats = AG.ConcatFunction.apply(el, pw)
            return feats if not return_weights else (feats, att_weights)
        feats = torch.empty((batch.shape[1], 2 * self.dim), dtype=torch.float32, device=self._dev())
        _, xprod = ops.gather_links(batch, X_node, want_sum=False, want_prod=True)
        self.elementwise_lin(xprod, out=feats[:, : self.dim])
        _, att_weights = self.calc_pairwise(batch, X_node, test_set, adj_mask=adj_mask, return_weights=return_weights,
                                            out=feats[:, self.dim:])
        return feats if not return_weights else (feats, att_weights)

    @_grad_if_training
    def propagate(self, adj=None, test_set=False):
        """reference :110-129 — GCN over the whole graph, then gnn_norm."""
        if adj is None:
            adj_norm = self.get_adj(test_set)
        else:
            adj_norm = gcn_normalise(csr_from_sparse(adj, self._dev()))   # caller-supplied graph: slow path
        x = self.data["x"]
        if "emb" in self.data:
            x = self.data["emb"](x)
        x = x.to(self._dev(), torch.float32)
        if not torch.is_grad_enabled():
            x = x.detach()
        # (gnn_norm rides in the epilogue of the last GCN layer's launch)
        return self.node_encoder(x, adj_norm, test_set, final_norm=(self.gnn_norm.weight, self.gnn_norm.bias))

    @torch.no_grad()
    def compute_node_mask(self, batch, test_set, adj):
        """reference :214-276, same return format: per type (ix int64 [2,S_t], src_ppr, tgt_ppr) or None.  In training
        mode with att_drop > 0 the sets are those left by node dropout (reference :257-260).  Its seed is the first draw
        from the CUDA generator, as in calc_pairwise, so after the same torch.manual_seed both keep the same pairs."""
        batch = ops.links_tensor(batch, self._dev())
        p_node = _drop_p(self, self.att_drop, batch)
        node_drop = (p_node, _seed(self, batch.device)) if p_node > 0 else None
        sel = self._select(batch, test_set, adj, want_link=True, node_drop=node_drop)
        res = []
        for t in range(3):
            produced = t == 0 or (t == 1 and self.mask != "cn") or (t == 2 and self.mask == "all")
            if not produced:
                res.append(None)
                continue
            r0, r1 = sel.type_range(t)
            ix = torch.stack((sel.link[r0:r1].long(), sel.node[r0:r1].long()))
            res.append((ix, sel.src_ppr[r0:r1], sel.tgt_ppr[r0:r1]))
        return tuple(res)

    def _select(self, batch, test_set, adj_mask=None, want_link=False, node_drop=None):
        """The selected pairs of the batch; node_drop = (p, seed): then only the pairs node dropout keeps (reference
        drop_pairwise :322-337: ceil(S (1 - p)) of them, after the >1-hop set is merged in)."""
        sel = self._select_all(batch, test_set, adj_mask, want_link)
        return sel if node_drop is None else ops.drop_pairs(sel, *node_drop)

    def _select_all(self, batch, test_set, adj_mask, want_link):
        stored = self.get_adj(test_set, mask=True)
        th = (self.thresh_cn, self.thresh_1hop, self.thresh_non1hop)
        if adj_mask is None:
            return ops.select(batch, stored, self.get_ppr(test_set), *th, self.mask, want_link=want_link)
        # A caller-supplied adjacency (the reference's training loop passes the graph with the batch's positives
        # removed) decides the CN and 1-hop sets only; the >1-hop set always comes from the STORED adjacency
        # (reference get_non_1hop_ppr :434-447 calls get_adj itself).  Slow path: the CSR is rebuilt per call.
        adj = csr_from_sparse(adj_mask, self._dev(), mask=True)
        if self.mask != "all":
            return ops.select(batch, adj, self.get_ppr(test_set), *th, self.mask, want_link=want_link)
        near = ops.select(batch, adj, self.get_ppr(test_set), *th, "1-hop", want_link=want_link)
        far = ops.select(batch, stored, self.get_ppr(test_set), *th, "all", want_link=want_link)
        return ops.merge_selections(near, far)

    @_grad_if_training
    def calc_pairwise(self, batch, X_node, test_set=False, adj_mask=None, return_weights=False, out=None):
        """reference :132-178.  Returns (pairwise feats [BS, dim], att_weights [2,S] or None).

        Links whose three node sets are all empty share one pairwise vector (attention output = LayerNorm(bias),
        counts = 0), so the attention + pairwise_lin stack runs only on the compacted list of non-empty links
        and the constant row is broadcast to the rest.

        Training mode: node dropout (att_drop) of the selected pairs, and dropout of each attention layer's output
        (layer.dropout; mask (seed, SITE_ATT + layer), row = batch position).  One seed per call, drawn first (see
        compute_node_mask).  With attention dropout every link gets its own masked row, so the stack runs on all links."""
        dev = self._dev()
        batch = ops.links_tensor(batch, dev)
        p_node = _drop_p(self, self.att_drop, batch, X_node)
        p_att = tuple(_drop_p(layer, layer.dropout, batch, X_node) for layer in self.att_layers)
        seed = _seed(self, dev) if p_node > 0 or any(p_att) else None
        X_node = self._check_x(X_node)
        bs = batch.shape[1]
        sel = self._select(batch, test_set, adj_mask, want_link=return_weights,
                           node_drop=(p_node, seed) if p_node > 0 else None)
        drop = (p_att, seed) if any(p_att) else None
        nnz = sel.nz.numel()
        if torch.is_grad_enabled():
            return self._pairwise_differentiable(batch, X_node, sel, return_weights, drop)
        if return_weights or nnz == bs or bs == 0 or drop is not None:
            pw, alpha = self._pairwise_rows(batch, X_node, sel, None, out=out, want_alpha=return_weights, drop=drop)
        else:
            alpha = None
            pw = out if out is not None else torch.empty((bs, self.dim), dtype=torch.float32, device=dev)
            rows = self._pairwise_rows(batch, X_node, sel, sel.nz)[0] if nnz > 0 else None
            ops.scatter_rows(rows, sel.nz, pw, fill_row=self._pw_const(X_node))
        att_weights = None
        if return_weights:
            att_weights = torch.stack((sel.link.float(), alpha))
        return pw, att_weights

    def _check_x(self, X_node):
        if not X_node.is_cuda:
            raise LpfError("X_node must be a CUDA tensor")
        if not torch.is_grad_enabled():
            X_node = X_node.detach()
        if X_node.dtype != torch.float32 or X_node.stride(-1) != 1:
            X_node = X_node.float().contiguous()
        return X_node

    def _pairwise_differentiable(self, batch, X_node, sel, return_weights, drop=None):
        """calc_pairwise with autograd (training mode): without attention dropout the empty-set links share one pairwise
        row, built through the attention bias -> LayerNorm -> pairwise_lin chain once, whose gradient is the sum over
        those links."""
        bs, nnz = sel.bs, sel.nz.numel()
        params = AG.pairwise_params(self)
        alpha = None
        if return_weights or nnz == bs or bs == 0 or drop is not None:
            res = AG.PairwiseFunction.apply(X_node, self, batch, sel, None, return_weights, drop, *params)
            feats, alpha = res if return_weights else (res, None)
            pw = self.pairwise_lin(feats)
        else:
            rows = None
            if nnz > 0:
                rows = self.pairwise_lin(AG.PairwiseFunction.apply(X_node, self, batch, sel, sel.nz, False, None,
                                                                   *params))
            pw = AG.ScatterFillFunction.apply(rows, self._pw_const_differentiable(X_node, params), sel.nz, bs)
        att_weights = torch.stack((sel.link.float(), alpha)) if return_weights else None
        return pw, att_weights

    def _empty_selection(self):
        dev = self._dev()
        return ops.Selection(self.mask, 1, torch.zeros(4, dtype=torch.int64, device=dev),
                             torch.empty(0, dtype=torch.int32, device=dev), torch.empty(0, device=dev),
                             torch.empty(0, device=dev), None, (0, 0, 0, 0), torch.empty(0, dtype=torch.int32, device=dev))

    def _pw_const_differentiable(self, X_node, params):
        """[1, dim] pairwise row of a link with empty node sets, with its autograd graph (built per call: a cached row
        would carry a graph that the first backward frees)."""
        empty = torch.zeros((2, 1), dtype=torch.int64, device=self._dev())
        return self.pairwise_lin(AG.PairwiseFunction.apply(X_node, self, empty, self._empty_selection(), None, False,
                                                           None, *params))

    def _pairwise_rows(self, batch, X_node, sel, idx, out=None, want_alpha=False, drop=None):
        """RPE -> attention layers -> counts -> pairwise_lin for the batch positions in idx (all links when None).
        Returns ([n, dim] rows in idx order, per-pair attention weights or None)."""
        feats, alpha, _ = self._attention_stack(batch, X_node, sel, idx, want_alpha, drop=drop)
        return self.pairwise_lin(feats, out=out), alpha

    def _attention_stack(self, batch, X_node, sel, idx, want_alpha=False, save=False, drop=None):
        """RPE -> attention layers -> counts for the batch positions in idx (all links when None): ([n, H*C +
        count_dim] rows in idx order, per-pair attention weights or None, and with save=True what the backward reads).
        drop = ((p of each layer), seed): each layer's [n, H*C] output is dropped before it feeds the next layer (mask
        rows are batch positions, so idx must be None)."""
        if drop is not None and idx is not None:
            raise ValueError("attention dropout runs over every link of the batch (idx must be None)")
        dev = self._dev()
        d, H = self.dim, self.num_heads
        n = sel.bs if idx is None else idx.numel()
        S = sel.total
        derived = self._get_derived()
        kvs = self._get_kv(X_node)

        # Pairs whose two PPR values are 0 see the RPE MLP at (0, 0): one row per node type instead of one per pair.  On
        # dense graphs with thresh_cn = 0 (ogbl-ddi shape: 285 common neighbours per link, 45 PPR entries per row) that
        # is most of the pairs, so large batches compute R only for the others and hand K4 a row map.  (Two more host
        # reads on this host-sized path; the rows are bit-identical either way: every row of rpe_hidden / gemm_tc is
        # computed on its own.)
        r_map = r_const = None
        pa, pb, bounds = sel.src_ppr, sel.tgt_ppr, sel.bounds
        if S >= self.rpe_map_min_pairs:
            live = (pa != 0) | (pb != 0)
            keep = torch.nonzero(live).reshape(-1)                      # host read 1: its size
            if keep.numel() <= S // 2:
                cb = torch.searchsorted(keep, torch.tensor(bounds, dtype=torch.int64, device=dev)).tolist()   # host read 2
                r_map = torch.cumsum(live, 0, dtype=torch.int32) - 1
                for t in range(3):
                    r0, r1 = bounds[t], bounds[t + 1]
                    if r1 > r0:
                        r_map[r0:r1].masked_fill_(~live[r0:r1], -1 - t)
                pa, pb, bounds = pa[keep].contiguous(), pb[keep].contiguous(), tuple(cb)
        Sc = bounds[3]
        csel = sel if r_map is None else ops.Selection(sel.mode, sel.bs, sel.ptr, sel.node, pa, pb, None, bounds, sel.nz)

        # RPE hidden vectors (shared by all layers)
        hsum = torch.empty((Sc, d), dtype=torch.float32, device=dev)
        for t, enc in enumerate(self._encoders()):
            ops.rpe_hidden(csel, t, enc.linears[0].weight, enc.linears[0].bias, enc.norm.weight, enc.norm.bias, hsum)
        if r_map is not None:       # the hidden vector of (0, 0), per type
            zsel = ops.Selection(sel.mode, 1, sel.ptr, sel.node, torch.zeros(3, device=dev), torch.zeros(3, device=dev), None,
                                 (0, 1, 2, 3), None)
            h0 = torch.zeros((3, d), dtype=torch.float32, device=dev)
            for t, enc in enumerate(self._encoders()):
                ops.rpe_hidden(zsel, t, enc.linears[0].weight, enc.linears[0].bias, enc.norm.weight, enc.norm.bias, h0)

        xsum, _ = ops.gather_links(batch, X_node, want_sum=True, want_prod=False, idx=idx)   # e1 + e2 of layer 0
        alpha = torch.empty(S, dtype=torch.float32, device=dev) if want_alpha else None
        feats = None
        st = {"csel": csel, "r_map": r_map, "hsum": hsum, "h0": h0 if r_map is not None else None, "kvs": kvs,
              "derived": derived, "Q": [], "R": [], "r_const": [], "feats_in": []} if save else None
        for l, layer in enumerate(self.att_layers):
            att = layer.att
            C = att.out_channels
            HC = H * C
            last = l == self.num_layers - 1
            if l == 0:
                Q = ops.linear(xsum, att.lin_l.weight, att.lin_l.bias, bias_scale=2.0)
            else:   # e1, e2 = chunk(2) of the previous layer's output (reference modules/layers.py:211)
                Q = ops.linear(feats, derived[l]["w_l_cat"], att.lin_l.bias, bias_scale=2.0)
            R = torch.empty((Sc, HC), dtype=torch.float32, device=dev)
            if r_map is not None:
                r_const = torch.zeros((3, HC), dtype=torch.float32, device=dev)
            for t, (m, c) in enumerate(derived[l]["rpe"]):
                r0, r1 = csel.type_range(t)
                if r1 > r0:
                    ops.linear(hsum[r0:r1], m, c, out=R[r0:r1])
                if r_map is not None:
                    ops.linear(h0[t:t + 1], m, c, out=r_const[t:t + 1])
            width = HC + (self.count_dim if last else 0)
            if save:
                st["Q"].append(Q)
                st["R"].append(R)
                st["r_const"].append(r_const)
                st["feats_in"].append(xsum if l == 0 else feats)
            feats = torch.empty((n, width), dtype=torch.float32, device=dev)
            ops.attend(sel, kvs[l], R, Q, att.att, att.bias, layer.post_att_norm.weight, layer.post_att_norm.bias,
                       H, C, write_counts=last, out=feats, alpha_out=alpha if last else None, idx=idx,
                       r_map=r_map, r_const=r_const)
            if drop is not None and drop[0][l] > 0:       # (not the counts)
                ops.dropout(feats[:, :HC], drop[0][l], drop[1], ops.SITE_ATT + l, out=feats[:, :HC])
        return feats, alpha, st

    def _node_tables(self, X_node, kv):
        """(X, KV) as the plan's kernels read them: the fp32 tensors, or bf16 copies built once per X_node."""
        if self.node_dtype != "bf16":
            return X_node, kv
        key = (X_node.data_ptr(), X_node._version, kv.data_ptr(), kv._version)
        if self._tab16 is None or self._tab16[0] != key:
            self._tab16 = (key, X_node.to(torch.bfloat16).contiguous(), kv.to(torch.bfloat16).contiguous())
        return self._tab16[1], self._tab16[2]

    def _pw_const(self, X_node):
        """[1, dim] pairwise vector of a link with empty node sets; depends on the weights only (cached)."""
        key = self._weights_key()
        if self._pw_const_cache is not None and self._pw_const_cache[0] == key:
            return self._pw_const_cache[1]
        dev = self._dev()
        row = self._pairwise_rows(torch.zeros((2, 1), dtype=torch.int64, device=dev), X_node, self._empty_selection(),
                                  None)[0]
        self._pw_const_cache = (key, row)
        return row

    # ------------------------------------------------------------------ fused eval body
    def _head_consts(self, score_func, X_node):
        """Operands of lpf_link_heads_tc (packed weights, folded pairwise constant), or None when the fused
        kernel does not cover this configuration."""
        d = self.dim
        if ops.GEMM_BACKEND != "tc" or d not in (32, 64) or self.num_layers != 1:
            return None
        if self.num_heads * self.att_layers[0].att.out_channels + self.count_dim > 256:
            return None          # the plan's contractions are single UMMA tiles (N <= 256): host-sized path instead
        lins = getattr(score_func, "lins", None)
        el = self.elementwise_lin
        if lins is None or len(lins) != 2 or tuple(lins[0].weight.shape) != (2 * d, 2 * d) or \
                tuple(lins[1].weight.shape) != (1, 2 * d) or len(el.linears) != 2 or el.norm is None:
            return None
        key = self._weights_key(score_func)
        if self._head_cache is not None and self._head_cache[0] == key:
            return self._head_cache[1]
        # no non-linearity between elementwise_lin's last Linear and mlp_score's first: fold them (fp64, once)
        ws1 = lins[0].weight.detach().double()
        w2, b2 = el.linears[1].weight.detach().double(), el.linears[1].bias.detach().double()
        w23 = (ws1[:, :d] @ w2).float().contiguous()
        consts = {
            "w1p": ops.pack_weight(el.linears[0].weight), "b1": el.linears[0].bias.detach().contiguous(),
            "ln_w": el.norm.weight.detach().contiguous(), "ln_b": el.norm.bias.detach().contiguous(),
            "w23": w23, "w23p": ops.pack_weight(w23), "ws1_pw": lins[0].weight.detach()[:, d:],
            "off": (ws1[:, :d] @ b2 + lins[0].bias.detach().double()).float().contiguous(),
            "ws2": lins[1].weight.detach().reshape(-1).contiguous(), "bs2": lins[1].bias.detach().contiguous(),
        }
        if d == 64 and ops.HEADS_F16:
            # operands of lpf_link_heads_f16: fp16 hi / lo images with exact power-of-two scales (see the header)
            import math
            sh = ops.pow2_scale(math.sqrt(d) * float(consts["ln_w"].abs().max()) + float(consts["ln_b"].abs().max()))
            consts["w1h"], sw1 = ops.pack_weight_f16(el.linears[0].weight)
            consts["w23h"], sw3 = ops.pack_weight_f16(w23)
            consts["inv_sw1"], consts["inv_s3"] = 1.0 / sw1, 1.0 / (sh * sw3)
            consts["ln_w_s"], consts["ln_b_s"] = (consts["ln_w"] * sh).contiguous(), (consts["ln_b"] * sh).contiguous()
        consts["c3"] = ops.linear(self._pw_const(X_node), consts["ws1_pw"], consts["off"]).reshape(-1).contiguous()
        self._head_cache = (key, consts)
        return consts

    @torch.no_grad()
    def score_links(self, batch, X_node, score_func, test_set=False, return_logits=False):
        """Body of the reference eval loops (train/testing.py:29-31, :113-115):
        score_func(cat(elementwise_lin(h[src]*h[dst]), calc_pairwise(...))).

        dim in {32, 64}: one fused tensor-core launch scores every link with the empty-set pairwise constant,
        then the (few) links with non-empty sets go through selection fill -> RPE -> attention -> pairwise_lin
        and are re-scored with their own pairwise vector."""
        dev = self._dev()
        X_node = self._check_x(X_node)
        consts = self._head_consts(score_func, X_node)
        if consts is None:
            batch = ops.links_tensor(batch, dev)
            feats = torch.empty((batch.shape[1], 2 * self.dim), dtype=torch.float32, device=dev)
            _, xprod = ops.gather_links(batch, X_node, want_sum=False, want_prod=True)
            self.elementwise_lin(xprod, out=feats[:, : self.dim])
            self.calc_pairwise(batch, X_node, test_set, out=feats[:, self.dim:])
            return score_func(feats, return_logits=return_logits) if return_logits else score_func(feats)
        plan = self._get_plan(score_func, consts, X_node, batch, test_set, return_logits)
        if plan is not None:
            prob, overflow = plan.run(batch)
            if not overflow:
                return prob.clone()
            self._plans.pop(plan.key, None)          # a pair pool was too small: host-sized path now, bigger pools next time
        batch = ops.links_tensor(batch, dev)
        bs = batch.shape[1]
        prob = torch.empty(bs, dtype=torch.float32, device=dev)
        ops.link_heads(batch, X_node, consts, prob, logits=return_logits)
        sel = self._select(batch, test_set)
        if plan is not None:
            self._plan_cap[plan.key] = 2 * max(b - a for a, b in zip(sel.bounds[:-1], sel.bounds[1:]))
        if sel.nz.numel() > 0:
            rows = self._pairwise_rows(batch, X_node, sel, sel.nz)[0]
            zb = ops.linear(rows, consts["ws1_pw"], consts["off"])
            ops.link_heads(batch, X_node, consts, prob, idx=sel.nz, zb=zb, logits=return_logits)
        return prob

    @torch.no_grad()
    def score_queries(self, source, targets, X_node, score_func, test_set=False, return_logits=False):
        """score_links for query groups: source [Q] and targets [Q, K] (both int32 or both int64, on the device or in
        pinned host memory) stand for the Q*K links (source[q], targets[q, j]) — the reference's citation2 eval input
        (train/testing.py:14-27: source.repeat(K) x negative targets).  Returns the [Q, K] scores.

        The groups are expanded into int64 links on the device (lpf_expand_query_links), so only 4 or 8 bytes per link
        and per query cross the host link instead of 16 per link.  A node id outside [0, num_nodes) raises LpfError."""
        source, targets = ops.query_groups(source, targets)
        X_node = self._check_x(X_node)
        dev = self._dev()
        Q, K = targets.shape
        if Q * K == 0:
            return torch.empty((Q, K), dtype=torch.float32, device=dev)
        links = torch.empty((2, Q * K), dtype=torch.int64, device=dev)
        bad = torch.zeros(1, dtype=torch.int64, device=dev)
        ops.expand_query_links(source.to(dev, non_blocking=True), targets.to(dev, non_blocking=True).reshape(-1), K, 0,
                               Q * K, self._id_bound(X_node, test_set), links, bad)
        prob = self.score_links(links, X_node, score_func, test_set=test_set, return_logits=return_logits)
        if int(bad.item()):                 # (score_links has already waited for the device)
            raise LpfError(f"query groups hold a node id outside [0, {self._id_bound(X_node, test_set)})")
        return prob.view(Q, K)

    def _id_bound(self, X_node, test_set):
        """Node ids index the rows of X_node and of the selection tables."""
        return min(X_node.shape[0], self.get_adj(test_set, mask=True).n, self.get_ppr(test_set).n)

    def _get_plan(self, score_func, consts, X_node, batch, test_set, logits):
        """The sync-free CUDA-graph plan for this batch size (plan.py), or None when the configuration needs the
        host-sized path (generic selection algorithm, i.e. a threshold of 0)."""
        if not self.use_plans or not torch.is_tensor(batch) or batch.dim() != 2 or batch.shape[0] != 2 or \
                batch.dtype != torch.int64 or batch.shape[1] == 0:
            return None
        adj, ppr = self.get_adj(test_set, mask=True), self.get_ppr(test_set)
        if ops.pick_select_algo(adj, ppr, self.thresh_1hop, self.thresh_non1hop, self.mask) == 0:
            return None
        key = (batch.shape[1], X_node.data_ptr(), X_node._version, bool(test_set), bool(logits), id(consts), self.node_dtype)
        plan = self._plans.get(key)
        if plan is None:
            from .plan import ScorePlan
            while len(self._plans) >= 2:                       # plans own capacity-sized buffers: keep two
                self._plans.pop(next(iter(self._plans)))
            plan = ScorePlan(self, score_func, consts, X_node, self._get_kv(X_node)[0], batch.shape[1], test_set, logits,
                             cap=self._plan_cap.get(key), use_graph=self.use_graphs)
            plan.key = key
            self._plans[key] = plan
        return plan
