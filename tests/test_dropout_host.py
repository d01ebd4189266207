"""CPU tests of dropout: the new header prototypes match the bindings, the entry points reject bad arguments, p outside
[0, 1] raises ValueError, CPU tensors with dropout > 0 in training mode raise NotImplementedError (before the CPU-tensor
LpfError), and eval mode never reaches a dropout op."""
import ctypes as C
import os
import re

import pytest
import torch

from oracle.golden import Golden

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DROPOUT = ("lpf_dropout", "lpf_gcn_layer_dropout", "lpf_layernorm_act_dropout", "lpf_drop_pairs_workspace_bytes",
           "lpf_drop_pairs_count", "lpf_drop_pairs_fill")


@pytest.fixture(scope="module")
def lib():
    from lpformer_b200.build import build
    build()
    from lpformer_b200 import _lib
    return _lib.load()


def _kind(ctype_name):
    return {"int": "i32", "int32_t": "i32", "int64_t": "i64", "float": "f", "double": "d", "void": None}.get(ctype_name, "p")


def test_dropout_prototypes_match_the_bindings(lib):
    from lpformer_b200 import _lib
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(REPO, "include", "lpformer_b200.h")).read(), flags=re.S)
    code = {C.c_int: "i32", C.c_int32: "i32", C.c_int64: "i64", C.c_float: "f", C.c_double: "d", C.c_void_p: "p"}
    for name in DROPOUT:
        m = re.search(r"\b(int|int64_t)\s+" + name + r"\s*\(([^)]*)\)", hdr)
        assert m, f"{name} is not declared"
        args = [a.strip() for a in m.group(2).split(",")]
        kinds = [k for k in ("p" if "*" in a else _kind(a.rsplit(" ", 1)[0].replace("const ", "").strip() if " " in a
                                                        else a) for a in args) if k is not None]
        res, argtypes = _lib.SIGNATURES[name]
        assert [code[t] for t in argtypes] == kinds, name
        assert code[res] == _kind(m.group(1)), name
        assert hasattr(lib, name)


def test_dropout_entry_points_validate_arguments(lib):
    seed = C.c_uint64(1)
    buf = (C.c_float * 16)()
    assert lib.lpf_dropout(buf, 4, buf, 4, 4, 4, 0, C.byref(seed), 1, 1.5, None) == -1
    assert b"p must be in [0, 1]" in lib.lpf_last_error()
    assert lib.lpf_dropout(buf, 4, buf, 4, 4, 4, 0, C.byref(seed), 1, -0.1, None) == -1
    assert lib.lpf_dropout(buf, 4, buf, 4, 4, 4, 0, None, 1, 0.5, None) == -1
    assert b"seed" in lib.lpf_last_error()
    assert lib.lpf_dropout(buf, 2, buf, 4, 4, 4, 0, C.byref(seed), 1, 0.5, None) == -1
    assert b"leading dimension" in lib.lpf_last_error()
    assert lib.lpf_dropout(None, 4, None, 4, 0, 4, 0, C.byref(seed), 1, 0.5, None) == 0      # no rows: nothing to do
    assert lib.lpf_layernorm_act_dropout(buf, 4, None, None, 0, 0, C.byref(seed), 1, 2.0, None, 0, buf, 4, 4, 4,
                                         None) == -1
    assert lib.lpf_gcn_layer_dropout(None, None, None, 0, 4, None, 4, None, 4, None, None, 0, C.byref(seed), 16, 0.5,
                                     None, 0, None, None, None, 4, None) == -1
    assert b"NULL" in lib.lpf_last_error()
    assert lib.lpf_drop_pairs_workspace_bytes() > 0
    assert lib.lpf_drop_pairs_count(None, 4, 10, 11, C.byref(seed), 2, None, None, 0, None) == -1
    assert b"K <= S" in lib.lpf_last_error()
    assert lib.lpf_drop_pairs_count(None, 4, 10, 5, C.byref(seed), 2, None, None, 0, None) == -1
    assert b"workspace" in lib.lpf_last_error()
    assert lib.lpf_drop_pairs_fill(None, 4, None, None, None, None, 10, C.byref(seed), 2, None, None, None, None, None,
                                   None, None) == -1


@pytest.mark.parametrize("p", [-0.1, 1.5, float("nan")])
def test_p_outside_the_unit_interval_raises(p):
    import lpformer_b200 as L
    from lpformer_b200 import ops
    with pytest.raises(ValueError):
        ops.check_p(p)
    with pytest.raises(ValueError):
        L.mlp_score(4, 4, 1, 2, dropout=p).train()(torch.zeros(3, 4))
    with pytest.raises(ValueError):
        L.MLP(2, 4, 4, 1, drop=p).train()(torch.zeros(3, 4))


def _model(name, train=True, **overrides):
    import lpformer_b200 as L
    g = Golden(name)
    targs = dict(g.train_args(), **overrides)
    model = L.LinkTransformer(targs, g.data_dict(), device="cpu")
    score = L.mlp_score(model.out_dim, model.out_dim, 1, 2)
    return g, model.train(train), score.train(train)


@pytest.mark.parametrize("grad", [True, False])
def test_cpu_tensors_with_dropout_raise_not_implemented(grad):
    """The masks exist on the device only: NotImplementedError, ahead of the LpfError of CPU tensors."""
    g, model, _ = _model("all_d32", feat_drop=0.2, gnn_drop=0.2, dropout=0.2, att_drop=0.2)
    links = torch.from_numpy(g["links"])
    with torch.set_grad_enabled(grad):
        for call in (lambda: model.propagate(), lambda: model.compute_node_mask(links, False, None),
                     lambda: model.calc_pairwise(links, torch.from_numpy(g["X_node"])),
                     lambda: __import__("lpformer_b200").mlp_score(4, 4, 1, 2, dropout=0.3).train()(torch.zeros(3, 4))):
            with pytest.raises(NotImplementedError, match="device only"):
                call()


def test_eval_mode_never_calls_a_dropout_op(monkeypatch):
    """Eval mode with every dropout > 0: no dropout entry point is reached (the forward fails on the CPU tensors
    further on, with LpfError, as every eval forward on the CPU does)."""
    from lpformer_b200 import _lib
    from lpformer_b200._lib import LpfError
    seen = []
    real = _lib.call

    def spy(name, *args, **kwargs):
        seen.append(name)
        return real(name, *args, **kwargs)
    monkeypatch.setattr(_lib, "call", spy)
    import lpformer_b200.ops as ops
    monkeypatch.setattr(ops, "call", spy)
    monkeypatch.setattr(ops, "draw_seed", lambda dev: pytest.fail("a dropout seed was drawn in eval mode"))
    g, model, score = _model("all_d32", train=False, feat_drop=0.3, gnn_drop=0.3, dropout=0.3, att_drop=0.3)
    model.elementwise_lin.dropout = 0.3
    links = torch.from_numpy(g["links"])
    for call in (lambda: model(links), lambda: model.compute_node_mask(links, False, None),
                 lambda: __import__("lpformer_b200").mlp_score(4, 4, 1, 2, dropout=0.3).eval()(torch.zeros(3, 4))):
        with pytest.raises(LpfError):
            call()
    assert not [n for n in seen if "drop" in n], seen
