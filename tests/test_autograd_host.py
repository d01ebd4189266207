"""CPU tests of the training path: dropout > 0 still raises in training mode, CPU tensors raise LpfError in training
mode too (no fallback), and the backward entry points of the header are bound with the argument lists _lib.py uses."""
import os
import re

import pytest
import torch

from oracle.golden import Golden

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BACKWARD = ("lpf_layernorm_act_backward", "lpf_gemm_wgrad", "lpf_act_backward", "lpf_gather_links_backward",
            "lpf_scatter_rows_backward", "lpf_rpe_hidden_backward", "lpf_attend_backward",
            "lpf_layernorm_act_backward_workspace_bytes", "lpf_gemm_wgrad_workspace_bytes",
            "lpf_scatter_rows_backward_workspace_bytes", "lpf_rpe_hidden_backward_workspace_bytes")


@pytest.fixture(scope="module")
def lib():
    from lpformer_b200.build import build
    build()
    from lpformer_b200 import _lib
    return _lib.load()


def _arity(ctype_name):
    return {"int": "i32", "int32_t": "i32", "int64_t": "i64", "float": "f"}.get(ctype_name, "p")   # (int is int32 here)


def test_backward_prototypes_match_the_bindings(lib):
    import ctypes as C
    from lpformer_b200 import _lib
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(REPO, "include", "lpformer_b200.h")).read(), flags=re.S)
    code = {C.c_int: "i32", C.c_int32: "i32", C.c_int64: "i64", C.c_float: "f", C.c_void_p: "p"}
    for name in BACKWARD:
        m = re.search(r"\b(int|int64_t)\s+" + name + r"\s*\(([^)]*)\)", hdr)
        assert m, f"{name} is not declared"
        args = [a.strip() for a in m.group(2).split(",")]
        kinds = ["p" if "*" in a else _arity(a.rsplit(" ", 1)[0].replace("const ", "").strip()) for a in args]
        res, argtypes = _lib.SIGNATURES[name]
        assert [code[t] for t in argtypes] == kinds, name
        assert code[res] == _arity(m.group(1)), name
        assert hasattr(lib, name)


def test_backward_entry_points_validate_arguments(lib):
    assert lib.lpf_gemm_wgrad(None, 4, None, 4, 4, 4, 4, None, 4, None, 0, None, 0, None) == -1
    assert b"no output" in lib.lpf_last_error()
    assert lib.lpf_layernorm_act_backward(None, 4, None, None, 0, None, 4, None, 4, 0, None, None, 0, 4, 2000, None, 0,
                                          None) == -1
    assert lib.lpf_attend_backward(None, 4, None, 4, None, None, 0, None, 0, None, None, None, 0, None, None, None, None,
                                   1, 32, None, 0, None, 0, None, None, 0, None, 0, None, None) == -1
    assert lib.lpf_rpe_hidden_backward_workspace_bytes(10, 32) > 0
    assert lib.lpf_gemm_wgrad_workspace_bytes(-1, 4, 4) == -1


def _model(name, train=True, **overrides):
    import lpformer_b200 as L
    g = Golden(name)
    targs = dict(g.train_args(), **overrides)
    model = L.LinkTransformer(targs, g.data_dict(), device="cpu")
    score = L.mlp_score(model.out_dim, model.out_dim, 1, 2)
    return g, model.train(train), score.train(train)


@pytest.mark.parametrize("what", ["dropout", "gnn_drop", "feat_drop", "att_drop"])
def test_dropout_still_raises_in_training_mode(what):
    g, model, _ = _model("all_d32", **{what: 0.1})
    links = torch.from_numpy(g["links"])
    with pytest.raises(NotImplementedError):
        if what == "dropout":
            model.elementwise_lin.dropout = 0.1
            model.elementwise_lin(torch.zeros(4, model.dim))
        elif what in ("gnn_drop", "feat_drop"):
            model.propagate()
        else:
            model.compute_node_mask(links, False, None)
    with pytest.raises(NotImplementedError):
        L_score = __import__("lpformer_b200").mlp_score(4, 4, 1, 2, dropout=0.5).train()
        L_score(torch.zeros(3, 4))


def test_cpu_tensors_raise_in_training_mode():
    from lpformer_b200._lib import LpfError
    g, model, score = _model("all_d32")
    assert torch.is_grad_enabled()
    links = torch.from_numpy(g["links"])
    with pytest.raises(LpfError):
        model(links)
    with pytest.raises(LpfError):
        model.propagate()
    with pytest.raises(LpfError):
        model.elementwise_lin(torch.zeros(4, model.dim, requires_grad=True))
    with pytest.raises(LpfError):
        score(torch.zeros(4, model.out_dim, requires_grad=True))
    with pytest.raises(LpfError):
        model.calc_pairwise(links, torch.from_numpy(g["X_node"]))
