"""ctypes binding of the C-ABI in include/lpformer_b200.h.

There is deliberately no fallback: if the shared library is missing or a call fails the
caller gets an exception.  Nothing in this package imports `oracle/`.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LPF_LIB_PATH") or os.path.join(_HERE, "_C", "liblpformer_b200.so")   # (override: A/B builds in development)

MODE = {"cn": 0, "1-hop": 1, "all": 2}
EPI_NONE, EPI_RELU, EPI_SIGMOID = 0, 1, 2
ALGO_GENERIC, ALGO_INTERSECT8, ALGO_INTERSECT32, ALGO_PACKED = 0, 1, 2, 3

_p, _i64, _i32, _f32, _int = C.c_void_p, C.c_int64, C.c_int32, C.c_float, C.c_int
_f64 = C.c_double

# name -> (restype, argtypes); mirrors include/lpformer_b200.h line by line
SIGNATURES = {
    "lpf_abi_version": (_int, []),
    "lpf_last_error": (C.c_char_p, []),
    "lpf_device_ok": (_int, []),
    "lpf_select_count": (_int, [_p, _i64, _p, _p, _p, _p, _p, _f32, _f32, _f32, _int, _int, _p, _p, _p]),
    "lpf_select_workspace_bytes": (_i64, [_i64]),
    "lpf_scan_scratch_bytes": (_i64, [_i64]),
    "lpf_scan_counts": (_int, [_p, _i64, _p, _p, _p]),
    "lpf_select_fill": (_int, [_p, _i64, _p, _p, _p, _p, _p, _f32, _f32, _f32, _int, _int, _p, _p, _p, _p, _p, _p,
                                _p]),
    "lpf_rpe_hidden": (_int, [_p, _p, _i64, _i64, _p, _p, _p, _p, _i32, _p, _i64, _p, _p]),
    "lpf_select_onepass": (_int, [_p, _i64, _p, _p, _p, _p, _p, _f32, _f32, _f32, _int, _int, _i64, _p, _p, _p, _p, _p,
                                  _p, _p, _p, _p]),
    "lpf_link_rows_bytes": (_i64, [_i64, _i64, _i64]),
    "lpf_link_rows_slab_bytes": (_i64, [_i64]),
    "lpf_link_rows_scratch_bytes": (_i64, [_i64]),
    "lpf_pack_link_rows": (_int, [_p, _p, _p, _p, _p, _i64, _p, _p, _p, _p]),
    "lpf_select_onepass_packed": (_int, [_p, _i64, _p, _p, _p, _p, _p, _p, _p, _f32, _f32, _f32, _int, _i64, _p, _p, _p,
                                         _p, _p, _p, _p, _p, _p]),
    "lpf_gemm": (_int, [_p, _i64, _p, _i64, _p, _f32, _p, _i64, _i64, _i32, _i32, _int, _p]),
    "lpf_pack_weight_bytes": (_i64, [_i32, _i32]),
    "lpf_pack_weight": (_int, [_p, _i64, _i32, _i32, _p, _p]),
    "lpf_gemm_tc": (_int, [_p, _i64, _p, _p, _f32, _p, _i64, _i64, _i32, _i32, _int, _p, _p]),
    "lpf_layernorm_act": (_int, [_p, _i64, _p, _p, _p, _i64, _p, _i64, _i64, _i32, _int, _p, _p]),
    "lpf_gather_links": (_int, [_p, _i64, _p, _i64, _p, _i64, _i32, _p, _i64, _p, _i64, _p, _int, _p]),
    "lpf_expand_query_links": (_int, [_p, _p, _i32, _i64, _i64, _i64, _i64, _p, _i64, _p, _p]),
    "lpf_expand_source_sweep": (_int, [_p, _i32, _i64, _i64, _i64, _i64, _p, _i64, _p, _p]),
    "lpf_topk_fold_workspace_bytes": (_i64, [_i64, _i32, _i64]),
    "lpf_topk_fold": (_int, [_p, _i64, _i64, _p, _p, _i32, _i64, _i64, _p, _p, _i64, _p, _i32, _p, _p, _p, _p, _p, _p,
                             _i64, _p]),
    "lpf_scatter_rows": (_int, [_p, _i64, _p, _i64, _p, _i64, _i64, _i32, _p, _p]),
    "lpf_debug_heads_clocks": (_int, [_p]),
    "lpf_debug_select_clocks": (_int, [_p]),
    "lpf_debug_select_timing": (_int, [_int]),
    "lpf_debug_select_slots": (_int, [_int]),
    "lpf_debug_select_timing_read": (_int, [_p]),
    "lpf_debug_nz_timing_read": (_int, [_p]),
    "lpf_select_compact": (_int, [_p, _i64, _p, _p, _p]),
    "lpf_link_heads_tc": (_int, [_p, _i64, _p, _i64, _p, _i64, _i32, _p, _p, _p, _p, _p, _p, _p, _i64, _p, _p,
                                 _p, _int, _p, _p, _p]),
    "lpf_pack_weight_f16_bytes": (_i64, [_i32, _i32]),
    "lpf_pack_weight_f16": (_int, [_p, _i64, _i32, _i32, _f32, _p, _p]),
    "lpf_link_heads_f16": (_int, [_p, _i64, _p, _i64, _p, _int, _i64, _i64, _i32, _p, _f32, _p, _p, _p, _p, _f32, _p, _p, _i64, _p, _p,
                                  _p, _int, _p, _p]),
    "lpf_debug_heads_f16_clocks": (_int, [_p]),
    "lpf_attend_fused": (_int, [_p, _i64, _p, _i64, _p, _p, _i64, _p, _i64, _p, _i64, _p, _p, _p, _p, _i32, _i32, _int, _int,
                                _p, _i64, _p, _p, _p, _p, _i64, _int, _p]),
    "lpf_attend_fused_ws": (_int, [_p, _i64, _p, _i64, _p, _p, _i64, _p, _i64, _p, _i64, _p, _p, _p, _p, _i32, _i32, _int, _int,
                                   _p, _i64, _p, _p, _p, _p, _i64, _int, _p, _p, _p, _i64, _p]),
    "lpf_attend_workspace_min": (_i64, []),
    "lpf_ppr_push_host": (_p, [_p, _p, _i64, C.c_double, C.c_double, _int, _p]),
    "lpf_ppr_push_slots": (_i32, [C.c_double, C.c_double]),
    "lpf_ppr_push_scratch_bytes": (_i64, [_i32, _i32]),
    "lpf_ppr_push": (_int, [_p, _p, _i64, C.c_double, C.c_double, _i64, _i64, _p, _p, _i32, _i32, _p, _p, _p, _p, _i64, _p, _p, _p]),
    "lpf_ppr_push_host_fetch": (_int, [_p, _p, _p, _p]),
    "lpf_gcn_spmm": (_int, [_p, _p, _p, _i64, _i64, _p, _i64, _p, _i32, _p, _i64, _p]),
    "lpf_gcn_layer": (_int, [_p, _p, _p, _i64, _i64, _p, _i64, _p, _i32, _p, _p, _int, _p, _i64, _p, _p, _p, _i64, _p]),
    # backward pass (csrc/backward.cu)
    "lpf_layernorm_act_backward_workspace_bytes": (_i64, [_i64, _i32]),
    "lpf_layernorm_act_backward": (_int, [_p, _i64, _p, _p, _int, _p, _i64, _p, _i64, _int, _p, _p, _int, _i64, _i32, _p,
                                          _i64, _p]),
    "lpf_gemm_wgrad_workspace_bytes": (_i64, [_i64, _i32, _i32]),
    "lpf_gemm_wgrad": (_int, [_p, _i64, _p, _i64, _i64, _i32, _i32, _p, _i64, _p, _int, _p, _i64, _p]),
    "lpf_act_backward": (_int, [_p, _i64, _p, _i64, _p, _i64, _i64, _i32, _int, _p]),
    "lpf_gather_links_backward": (_int, [_p, _i64, _p, _i64, _p, _i64, _i32, _p, _i64, _p, _i64, _p, _i64, _p]),
    "lpf_scatter_rows_backward_workspace_bytes": (_i64, [_i64, _i32]),
    "lpf_scatter_rows_backward": (_int, [_p, _i64, _i64, _i32, _p, _i64, _p, _i64, _p, _p, _i64, _p]),
    "lpf_rpe_hidden_backward_workspace_bytes": (_i64, [_i64, _i32]),
    "lpf_rpe_hidden_backward": (_int, [_p, _p, _i64, _i64, _p, _p, _p, _p, _i32, _p, _i64, _p, _p, _p, _p, _int, _p, _i64,
                                       _p]),
    "lpf_attend_backward": (_int, [_p, _i64, _p, _i64, _p, _p, _i64, _p, _i64, _p, _p, _p, _i64, _p, _p, _p, _p, _i32,
                                   _i32, _p, _i64, _p, _i64, _p, _p, _i64, _p, _i64, _p, _p]),
    # dropout (csrc/dropout.cu, spmm.cu, dense.cu)
    "lpf_dropout": (_int, [_p, _i64, _p, _i64, _i64, _i32, _i64, _p, _i32, _f64, _p]),
    "lpf_gcn_layer_dropout": (_int, [_p, _p, _p, _i64, _i64, _p, _i64, _p, _i32, _p, _p, _int, _p, _i32, _f64, _p, _i64,
                                     _p, _p, _p, _i64, _p]),
    "lpf_layernorm_act_dropout": (_int, [_p, _i64, _p, _p, _int, _i64, _p, _i32, _f64, _p, _i64, _p, _i64, _i64, _i32,
                                         _p]),
    "lpf_drop_pairs_workspace_bytes": (_i64, []),
    "lpf_drop_pairs_count": (_int, [_p, _i64, _i64, _i64, _p, _i32, _p, _p, _i64, _p]),
    "lpf_drop_pairs_fill": (_int, [_p, _i64, _p, _p, _p, _p, _i64, _p, _i32, _p, _p, _p, _p, _p, _p, _p]),
}



class NzArgs(C.Structure):
    """lpf_nz_args of include/lpformer_b200.h (field order and types must match)."""
    _fields_ = ([("links", _p), ("bs", _i64), ("nz", _p), ("n_cap", _i64), ("n_dev", _p), ("X", _p), ("ldx", _i64),
                 ("KV", _p), ("ld_kv", _i64), ("node", _p), ("src_ppr", _p), ("tgt_ppr", _p), ("seg_start", _p),
                 ("counts", _p), ("cap", _i64), ("header", _p), ("R", _p), ("d", _i32), ("mode", _i32), ("wlT", _p), ("bl", _p)] +
                [(n, _p * 3) for n in ("rpe_w1", "rpe_b1", "rpe_ln_w", "rpe_ln_b", "rpe_mT", "rpe_c")] +
                [(n, _p) for n in ("att", "att_bias", "post_ln_w", "post_ln_b", "p1T", "pb1", "pln_w", "pln_b", "p2T",
                                   "pb2", "wzT", "off", "w1T", "b1", "ln_w", "ln_b", "w23T", "ws2", "bs2", "prob")] +
                [("logits", _i32), ("tab_bf16", _i32)])


SIGNATURES["lpf_nz_links_fused"] = (_int, [C.POINTER(NzArgs), _p])
SIGNATURES["lpf_nz_pairs"] = (_int, [C.POINTER(NzArgs), _p])

_lib = None


class LpfError(RuntimeError):
    pass


def load():
    """Load (once) and return the ctypes library.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LpfError(
            f"{LIB_PATH} not found: build the sm_100a extension first (python -m lpformer_b200.build). "
            "lpformer_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


# kernels launched per entry point (for bench.py's gpu_launches and per-kernel CUDA-event timing)
KERNEL_LAUNCHES = {"lpf_select_count": 3, "lpf_scan_counts": 2, "lpf_select_fill": 2, "lpf_rpe_hidden": 1,
                   "lpf_gemm": 1, "lpf_gemm_tc": 1, "lpf_pack_weight": 1, "lpf_layernorm_act": 1, "lpf_gather_links": 1, "lpf_expand_query_links": 1, "lpf_expand_source_sweep": 1, "lpf_topk_fold": 2, "lpf_attend_fused": 1, "lpf_attend_fused_ws": 2,
                   "lpf_gcn_spmm": 1, "lpf_gcn_layer": 1, "lpf_nz_links_fused": 2, "lpf_nz_pairs": 1, "lpf_select_compact": 2, "lpf_select_onepass": 4, "lpf_select_onepass_packed": 6, "lpf_pack_link_rows": 4, "lpf_scatter_rows": 2, "lpf_link_heads_tc": 1, "lpf_link_heads_f16": 1, "lpf_pack_weight_f16": 1,
                   "lpf_gemm_wgrad": 2, "lpf_act_backward": 1, "lpf_gather_links_backward": 1,
                   "lpf_rpe_hidden_backward": 2, "lpf_attend_backward": 1,
                   "lpf_dropout": 1, "lpf_gcn_layer_dropout": 1, "lpf_layernorm_act_dropout": 1, "lpf_drop_pairs_count": 18,
                   "lpf_drop_pairs_fill": 1}   # (+ two counted per call: see ops.py)


class Trace:
    """Optional per-call instrumentation: counts launches and brackets every entry point with CUDA
    events on the launching stream.  Enabled by bench.py; off by default."""

    def __init__(self, events=True):
        self.events = events
        self.launches = 0
        self.records = []   # (name, meta, start_event, end_event)

    def summary(self):
        """name -> (calls, total_ms); call after torch.cuda.synchronize()."""
        out = {}
        for name, _, a, b in self.records:
            c, t = out.get(name, (0, 0.0))
            out[name] = (c + 1, t + a.elapsed_time(b))
        return out


TRACE = None
COUNTERS = None   # optional dict: bench.py counts CUDA-graph launches here


def call(name, *args, meta=None, label=None, launches=None):
    """Invoke an int-returning entry point; raise LpfError with lpf_last_error() on failure.  `label`: the tracer
    files the call under name/label (two uses of one entry point that should be timed apart).  `launches`: the kernels
    this call launches, for entry points whose count depends on their arguments (KERNEL_LAUNCHES otherwise)."""
    lib = load()
    tr = TRACE
    if tr is not None:
        tr.launches += KERNEL_LAUNCHES.get(name, 0) if launches is None else launches
        if tr.events:
            a = torch.cuda.Event(enable_timing=True)
            b = torch.cuda.Event(enable_timing=True)
            a.record()
            rc = getattr(lib, name)(*args)
            b.record()
            tr.records.append((name if label is None else name + "/" + label, meta, a, b))
        else:
            rc = getattr(lib, name)(*args)
    else:
        rc = getattr(lib, name)(*args)
    if rc != 0:
        raise LpfError(f"{name} failed ({rc}): {lib.lpf_last_error().decode()}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return t.data_ptr()


def stream():
    """The current torch CUDA stream as a void*."""
    return torch.cuda.current_stream().cuda_stream


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise LpfError("lpformer_b200 kernels need CUDA tensors (no CPU fallback); got a %s tensor" % t.device)
