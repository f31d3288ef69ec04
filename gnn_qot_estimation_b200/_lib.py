"""ctypes binding of libqot_b200.so (C ABI declared in include/qot_b200.h).

There is NO fallback: if the library is missing or cannot be loaded the import of
any compute op raises, and every op refuses non-CUDA tensors.
"""
from __future__ import annotations

import ctypes as C
import functools
from pathlib import Path

import torch

_PKG = Path(__file__).resolve().parent
import os as _os

# QOT_B200_LIB: developer override pointing at an instrumented build of the same sources
LIB_PATH = Path(_os.environ["QOT_B200_LIB"]) if _os.environ.get("QOT_B200_LIB") else _PKG / "libqot_b200.so"

_lib = None

i64, i32, f32p, vp, sz = C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_size_t
P = C.c_void_p  # every device pointer travels as an integer address


class QotStore(C.Structure):
    _fields_ = [("node_ptr", P), ("edge_ptr", P), ("edge_src", P), ("edge_dst", P),
                ("node_feat", P), ("edge_feat", P), ("y", P),
                ("node_dim", i32), ("edge_dim", i32), ("y_dim", i32)]


class QotLpGraphCfg(C.Structure):
    _fields_ = [("F", i32), ("L", i32), ("Q", i32), ("T", i32),
                ("i_conn", i32), ("i_osnr", i32), ("i_snr", i32), ("i_ber", i32),
                ("i_feat", i32 * 4), ("feat_lo", C.c_double * 4), ("feat_hi", C.c_double * 4),
                ("i_tgt", i32 * 3), ("tgt_lo", C.c_double * 3), ("tgt_hi", C.c_double * 3),
                ("freq_threshold", C.c_double)]


class QotLpState(C.Structure):
    _fields_ = [("cfg", QotLpGraphCfg), ("S", i64), ("N", i64), ("E", i64),
                ("freqs", P), ("x", P), ("node_ptr", P), ("rowptr", P), ("edge_index", P), ("chan_node", P),
                ("conn_ids", P)]


class QotLpChanges(C.Structure):
    _fields_ = [("K", i64), ("n_links", i64),
                ("node", P), ("sample", P), ("link_ptr", P), ("links", P), ("q0", P), ("width", P), ("feat", P)]


class QotLpDemands(C.Structure):
    _fields_ = [("D", i64), ("P", i64), ("n_links", i64),
                ("sample", P), ("opt_ptr", P), ("link_ptr", P), ("links", P), ("width", P), ("feat", P),
                ("own_bound", P)]


class QotLightpathParams(C.Structure):
    _fields_ = [("lin_w", P), ("att_src", P), ("att_dst", P), ("conv_bias", P),
                ("bn_w", P), ("bn_b", P), ("bn_mean", P), ("bn_var", P),
                ("mlp_w1", P), ("mlp_b1", P), ("mlp_w2", P), ("mlp_b2", P),
                ("bn_eps", C.c_float), ("is_lut_index", i32)]


class QotLpBatch(C.Structure):
    _fields_ = [("x", P), ("edge_index", P), ("ptr", P), ("edge_ptr", P), ("lut_ptr", P),
                ("N", i64), ("E", i64), ("B", i64),
                ("out", P), ("lut_batch", P), ("lut_node", P), ("n_lut", P), ("status", P), ("z", P),
                ("tile0", i64), ("reserved", i64)]


class QotParamSeg(C.Structure):
    _fields_ = [("param", P), ("offset", i64), ("numel", i64)]


class QotSgdHyper(C.Structure):
    _fields_ = [("lr", C.c_float), ("momentum", C.c_float), ("dampening", C.c_float), ("weight_decay", C.c_float),
                ("nesterov", i32), ("maximize", i32), ("one_minus_dampening", C.c_float), ("reserved", i32)]


class QotLpWireSlot(C.Structure):
    _fields_ = [("arena", P), ("x", P), ("edge_index", P), ("ptrs", P), ("desc", P), ("result", P),
                ("lut_node", P), ("n_lut", P),
                ("cap_nodes", i64), ("cap_edges", i64), ("cap_graphs", i64)]


# name -> (restype, argtypes); mirrors include/qot_b200.h one to one
SIGNATURES = {
    "qot_last_error": (C.c_char_p, []),
    "qot_version": (C.c_int, []),
    "qot_collate": (C.c_int, [C.POINTER(QotStore), P, i64, P, P, i64, i64, P, P, P, P, P, P, vp]),
    "qot_csr_workspace_bytes": (sz, [i64, i64]),
    "qot_build_csr": (C.c_int, [P, i64, i64, C.c_int, C.c_int, P, P, P, P, P, sz, vp]),
    "qot_graph_ptr": (C.c_int, [P, i64, i64, P, vp]),
    "qot_edge_ptr": (C.c_int, [P, i64, P, i64, i64, P, P, vp]),
    "qot_gemm": (C.c_int, [P, i64, i64, P, P, i64, i64, P, P, i64, i64, i64, i64, vp]),
    "qot_gemm_tf32x3_workspace_bytes": (sz, [i64, i64, i64]),
    "qot_debug_gemm_tiles": (i64, [i64, i64, i64, i64, i64, P, i64]),
    "qot_gemm_tf32x3": (C.c_int, [P, i64, P, P, i64, P, P, i64, i64, i64, i64, P, P, sz, vp]),
    "qot_wgrad_tf32x3_workspace_bytes": (sz, [i64, i64, i64]),
    "qot_wgrad_tf32x3": (C.c_int, [P, i64, P, i64, P, i64, i64, i64, P, i64, P, P, sz, vp]),
    "qot_wgrad_workspace_bytes": (sz, [i64, i64, i64]),
    "qot_wgrad": (C.c_int, [P, i64, P, i64, i64, i64, i64, P, i64, P, sz, vp]),
    "qot_colsum_workspace_bytes": (sz, [i64, i64]),
    "qot_colsum": (C.c_int, [P, i64, i64, i64, P, P, sz, vp]),
    "qot_segment_sum_workspace_bytes": (sz, [i64, i64, i64]),
    "qot_segment_sum": (C.c_int, [P, P, P, i64, i64, i64, P, P, sz, vp]),
    "qot_tconv_fwd": (C.c_int, [P, P, P, P, P, P, i64, i64, C.c_float, P, P, P, P, vp]),
    "qot_tconv_bwd_workspace_bytes": (sz, [i64, i64, i64]),
    "qot_tconv_bwd": (C.c_int, [P, P, P, P, P, P, P, P, P, P, P, P, P, P, i64, i64, i64,
                                C.c_float, P, P, P, sz, vp]),
    "qot_nnconv_fwd": (C.c_int, [P, P, P, P, P, P, P, P, i64, i64, C.c_float, P, vp]),
    "qot_nnconv_bwd_workspace_bytes": (sz, [i64, i64, i64]),
    "qot_nnconv_bwd": (C.c_int, [P, P, P, P, P, P, P, P, P, P, P, P, i64, i64, i64, C.c_float,
                                 P, P, P, P, P, sz, vp]),
    "qot_pool_mlp_fwd_workspace_bytes": (sz, [i64, i64, i64]),
    "qot_pool_mlp_fwd": (C.c_int, [P, P, i64, i64, i64, P, P, P, P, P, P, P, P, P, sz, vp]),
    "qot_pool_mlp_bwd_workspace_bytes": (sz, [i64, i64]),
    "qot_pool_mlp_bwd": (C.c_int, [P, P, P, P, P, i64, i64, i64, P, P, P, P, P, P, P, P, sz, vp]),
    "qot_lightpath_lut_ptr_workspace_bytes": (sz, [i64]),
    "qot_lightpath_lut_ptr": (C.c_int, [P, P, i64, i64, i32, P, P, sz, vp]),
    "qot_lightpath_prepared_floats": (sz, []),
    "qot_lightpath_prepare": (C.c_int, [C.POINTER(QotLightpathParams), P, vp]),
    "qot_lightpath_infer_workspace_bytes": (sz, [i64]),
    "qot_lightpath_graph_scratch_bytes": (sz, [i64]),
    "qot_lightpath_graph_count": (C.c_int, [P, P, P, i64, C.POINTER(QotLpGraphCfg), P, P, P, sz, P, vp]),
    "qot_lightpath_graph_fill": (C.c_int, [P, i64, P, P, P, P, P, P, P, vp]),
    "qot_lightpath_channel_map": (C.c_int, [P, i64, C.POINTER(QotLpGraphCfg), P, P, i64, P, P, vp]),
    "qot_lightpath_candidates": (C.c_int, [C.POINTER(QotLpState), C.POINTER(QotLpChanges), P, i32, i32, P, P, P, P, P,
                                           vp]),
    "qot_lightpath_reconfigure": (C.c_int, [C.POINTER(QotLpState), C.POINTER(QotLpChanges), P, i32, i32, P, P, P, P,
                                            P, P, vp]),
    "qot_lightpath_change_sets": (C.c_int, [C.POINTER(QotLpState), C.POINTER(QotLpChanges), i64, P, P, i32, i32, P, P,
                                            P, P, P, P, P, vp]),
    "qot_lightpath_placements": (C.c_int, [C.POINTER(QotLpState), C.POINTER(QotLpDemands), P, i32, i32, i32, P, i32,
                                           i32, P, P, P, P, P, P, P, P, P, P, P, P, vp]),
    "qot_lightpath_provision": (C.c_int, [C.POINTER(QotLpState), C.POINTER(QotLpDemands), P, P, P, i32, i32, i32, P,
                                          i32, i32, P, P, P, P, P, P, P, P, P, P, P, P, P, vp]),
    "qot_topological_graph_scratch_bytes": (sz, [i64]),
    "qot_topological_graph_count": (C.c_int, [P, P, i64, C.POINTER(QotLpGraphCfg), i32, i32, i32, P, P, P, sz, P, vp]),
    "qot_topological_graph_fill": (C.c_int, [P, i64, P, P, P, P, P, vp]),
    "qot_topo_fused_params": (C.c_int, []),
    "qot_topo_fused_prepared_floats": (C.c_int, []),
    "qot_topo_fused_prepare": (C.c_int, [P, P, vp]),
    "qot_topo_fused_saved_floats": (sz, [i64, i64, i64]),
    "qot_topo_fused_fwd": (C.c_int, [P, P, P, P, i64, P, P, P, i64, i64, i32, i32, i32, P, P, P, P, C.c_float, C.c_float, vp]),
    "qot_topo_fused_bwd_workspace_bytes": (sz, [i32]),
    "qot_topo_fused_bwd": (C.c_int, [P, P, P, P, i64, P, P, P, i64, i64, i32, i32, i32, P, P, P, P, P, sz, P, P, C.c_float,
                                     C.c_float, vp]),
    "qot_ddp_exchange_bytes": (sz, [i64]),
    "qot_ddp_sgd_step": (C.c_int, [P, P, i32, i32, i64, P, i32, P, P, P, P, vp]),
    "qot_lightpath_stream_tiles": (i64, [i64]),
    "qot_lightpath_infer_stream": (C.c_int, [P, i32, i64, i64, i64, P, i32, i32, vp]),
    "qot_lightpath_every_node_tiles": (i64, [i64]),
    "qot_lightpath_infer_every_node": (C.c_int, [P, i32, i64, i64, P, i32, i32, vp]),
    "qot_lightpath_wire_bytes": (sz, [i64, i64, i64, i64]),
    "qot_lightpath_wire_result_bytes": (sz, [i64]),
    "qot_lightpath_infer_wire_host": (C.c_int, [P, i64, i64, i64, i64, P, i32, C.POINTER(QotLpWireSlot), P,
                                                C.POINTER(i64), C.POINTER(i64), vp]),
    "qot_gat_fwd": (C.c_int, [P, P, P, i64, P, P, P, P, P, P, P, P, vp]),
    "qot_gat_bwd_workspace_bytes": (sz, [i64]),
    "qot_gat_bwd": (C.c_int, [P, P, P, i64, P, P, P, P, P, P, P, P, P, P, P, P, sz, vp]),
    "qot_bn_stats_workspace_bytes": (sz, [i64, i64]),
    "qot_bn_stats": (C.c_int, [P, i64, i64, P, P, P, P, C.c_float, P, sz, vp]),
    "qot_bn_apply": (C.c_int, [P, i64, i64, P, P, C.c_float, P, P, P, vp]),
    "qot_bn_bwd_dense_workspace_bytes": (sz, [i64, i64]),
    "qot_bn_bwd_dense": (C.c_int, [P, P, P, C.c_float, P, P, i64, i64, C.c_int, P, P, P, P, sz, vp]),
    "qot_mean_pool_workspace_bytes": (sz, [i64, i64, i64]),
    "qot_mean_pool_fwd": (C.c_int, [P, P, i64, i64, i64, P, P, sz, vp]),
    "qot_mean_pool_bwd": (C.c_int, [P, P, i64, i64, i64, P, P, sz, vp]),
    "qot_smooth_l1_workspace_bytes": (sz, [i64]),
    "qot_smooth_l1": (C.c_int, [P, P, P, i64, C.c_float, P, P, P, P, sz, vp]),
    "qot_lut_select_workspace_bytes": (sz, [i64]),
    "qot_lut_select": (C.c_int, [P, i64, i64, i32, P, P, P, P, P, sz, vp]),
    "qot_lut_head_fwd": (C.c_int, [P, P, i64, P, P, C.c_float, P, P, P, P, P, P, P, P, P, P, vp]),
    "qot_lut_head_bwd_workspace_bytes": (sz, [i64]),
    "qot_lut_head_bwd": (C.c_int, [P, P, P, P, i64, P, P, P, P, P, P, P, P, sz, vp]),
    "qot_bn_bwd_workspace_bytes": (sz, [i64, i64, i64]),
    "qot_bn_bwd_sparse": (C.c_int, [P, P, P, C.c_float, P, P, P, i64, i64, i64, C.c_int, P, P, P, P, sz, vp]),
}


def lib() -> C.CDLL:
    """Loads libqot_b200.so (once).  Raises loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m gnn_qot_estimation_b200.build` "
            "(nvcc, sm_100a).  gnn_qot_estimation_b200 has no CPU or PyTorch fallback.")
    handle = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(handle, name)   # AttributeError if the .so lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = handle
    return handle


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().qot_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libqot_b200 {what} failed (code {rc}): {msg}")


def ptr(t):
    """Device address of a tensor (None -> NULL).  Refuses anything not on CUDA."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("gnn_qot_estimation_b200 ops need CUDA tensors (no CPU fallback)")
    if not t.is_contiguous():
        raise RuntimeError("gnn_qot_estimation_b200 ops need contiguous tensors")
    return t.data_ptr()


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _device_of(args, kwargs):
    for a in list(args) + list(kwargs.values()):
        if torch.is_tensor(a):
            if a.is_cuda:
                return a.device
        elif not isinstance(a, torch.nn.Module):
            t = getattr(a, "edge_index", None)
            if torch.is_tensor(t) and t.is_cuda:
                return t.device
            d = getattr(a, "device", None)
            if isinstance(d, torch.device) and d.type == "cuda":
                return d
    return None


def on_tensor_device(fn):
    """Runs `fn` with the device of its first CUDA tensor (or batch / store) argument current, so that
    `stream()`, workspaces and every `cudaFuncSetAttribute` inside the library refer to the GPU the data
    lives on -- a process may drive several GPUs (one process per GPU is the normal deployment)."""
    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        dev = _device_of(args, kwargs)
        if dev is None or dev.index is None or dev.index == torch.cuda.current_device():
            return fn(*args, **kwargs)
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)
    return wrapper


_ws_cache = {}


def workspace(nbytes: int, device) -> torch.Tensor:
    """A per-(device, stream) scratch buffer that only grows.  Kernels on one stream
    run in order, so reusing it between calls is safe."""
    key = (device.index if device.index is not None else torch.cuda.current_device(),
           torch.cuda.current_stream(device).cuda_stream)
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
        _ws_cache[key] = buf
    return buf
