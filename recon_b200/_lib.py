"""ctypes binding of libspkbgat.so (the C ABI declared in include/spkbgat.h).

There is no CPU fallback: importing the ops without the built library, or calling them without a
CUDA device, raises. The library is built in-tree by `__graft_entry__.build()` /
`make -C recon_b200/csrc`.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SPK_LIB") or os.path.join(_HERE, "libspkbgat.so")     # SPK_LIB: A/B builds of the same ABI

c_i32p = C.POINTER(C.c_int32)
c_i64p = C.POINTER(C.c_int64)
c_f32p = C.POINTER(C.c_float)
ABI_VERSION = 6


class Geom(C.Structure):
    _fields_ = [("n_heads", C.c_int32), ("d_head", C.c_int32), ("d_pad", C.c_int32), ("width", C.c_int32)]


class HubTasks(C.Structure):
    _fields_ = [("task_seg", C.c_void_p), ("task_beg", C.c_void_p), ("task_end", C.c_void_p),
                ("hub_seg", C.c_void_p), ("hub_task_ptr", C.c_void_p),
                ("partial", C.c_void_p), ("ldpart", C.c_int64),
                ("n_tasks", C.c_int32), ("n_hubs", C.c_int32), ("hub_thresh", C.c_int32), ("reserved", C.c_int32),
                ("task_order", C.c_void_p)]


class EdgeFwdArgs(C.Structure):
    _fields_ = [("segptr", C.c_void_p), ("col", C.c_void_p), ("t1", C.c_void_p), ("t2", C.c_void_p),
                ("P1", C.c_void_p), ("ld1", C.c_int64), ("P2", C.c_void_p), ("ld2", C.c_int64),
                ("P3", C.c_void_p), ("ld3", C.c_int64),
                ("mask", C.c_void_p), ("mask_stride", C.c_int64),
                ("out", C.c_void_p), ("ldo", C.c_int64), ("den", C.c_void_p), ("sw", C.c_void_p),
                ("nanflag", C.c_void_p),
                ("n_rows", C.c_int32), ("apply_elu", C.c_int32), ("alpha", C.c_float), ("elu_rows", C.c_int32),
                ("geom", Geom), ("hub", HubTasks)]


class EdgeBwdRowsArgs(C.Structure):
    _fields_ = [("segptr", C.c_void_p), ("col", C.c_void_p), ("t1", C.c_void_p), ("t2", C.c_void_p),
                ("P1", C.c_void_p), ("ld1", C.c_int64), ("P2", C.c_void_p), ("ld2", C.c_int64),
                ("P3", C.c_void_p), ("ld3", C.c_int64),
                ("mask", C.c_void_p), ("mask_stride", C.c_int64),
                ("out", C.c_void_p), ("dout", C.c_void_p), ("ldo", C.c_int64),
                ("den", C.c_void_p),
                ("G", C.c_void_p), ("ldg", C.c_int64), ("dP1", C.c_void_p), ("ldd1", C.c_int64),
                ("rec", C.c_void_p),
                ("n_rows", C.c_int32), ("apply_elu", C.c_int32), ("alpha", C.c_float), ("reserved", C.c_int32),
                ("geom", Geom), ("hub", HubTasks)]


class SegGatherArgs(C.Structure):
    _fields_ = [("segptr", C.c_void_p), ("src", C.c_void_p), ("pos", C.c_void_p),
                ("G", C.c_void_p), ("ldg", C.c_int64), ("rec", C.c_void_p),
                ("out", C.c_void_p), ("ldout", C.c_int64),
                ("n_seg", C.c_int32), ("flags", C.c_int32),
                ("geom", Geom), ("hub", HubTasks)]


class EdgeBwdFusedArgs(C.Structure):
    _fields_ = [("rowptr", C.c_void_p),
                ("colptr", C.c_void_p), ("csc_row", C.c_void_p), ("csc_pos", C.c_void_p), ("csc_t1", C.c_void_p),
                ("csc_t2", C.c_void_p),
                ("P1", C.c_void_p), ("ld1", C.c_int64), ("P2", C.c_void_p), ("ld2", C.c_int64),
                ("P3", C.c_void_p), ("ld3", C.c_int64),
                ("mask", C.c_void_p), ("mask_stride", C.c_int64),
                ("out", C.c_void_p), ("dout", C.c_void_p), ("ldo", C.c_int64),
                ("den", C.c_void_p), ("sw", C.c_void_p),
                ("G", C.c_void_p), ("ldg", C.c_int64), ("rowsc", C.c_void_p),
                ("dP1", C.c_void_p), ("ldd1", C.c_int64), ("dP2", C.c_void_p), ("ldd2", C.c_int64),
                ("rec", C.c_void_p),
                ("n_rows", C.c_int32), ("n_cols", C.c_int32), ("apply_elu", C.c_int32), ("alpha", C.c_float),
                ("geom", Geom), ("row_hub", HubTasks), ("col_hub", HubTasks)]


class EdgeBwdSplitArgs(C.Structure):
    _fields_ = [("base", EdgeBwdFusedArgs),
                ("relptr", C.c_void_p), ("rel_row", C.c_void_p), ("rel_pos", C.c_void_p),
                ("rec4", C.c_void_p), ("dsv", C.c_void_p),
                ("dP3", C.c_void_p), ("ldd3", C.c_int64),
                ("n_rel", C.c_int32), ("phases", C.c_int32),
                ("rel_hub", HubTasks),
                ("colsum", C.c_void_p), ("ld_colsum", C.c_int64),
                ("rowsum", C.c_void_p), ("ld_rowsum", C.c_int64),
                ("G_rel", C.c_void_p), ("ldg_rel", C.c_int64),
                ("dup", C.c_int32), ("reserved", C.c_int32)]


class AggGeom(C.Structure):
    _fields_ = [("n_heads", C.c_int32), ("f_chunks", C.c_int32), ("r_chunks", C.c_int32), ("lz", C.c_int32)]


class AggFwdArgs(C.Structure):
    _fields_ = [("segptr", C.c_void_p), ("col", C.c_void_p), ("t1", C.c_void_p), ("t2", C.c_void_p),
                ("xrow", C.c_void_p), ("ldxr", C.c_int64), ("xcol", C.c_void_p), ("ldxc", C.c_int64),
                ("rel", C.c_void_p), ("ldr", C.c_int64),
                ("mask", C.c_void_p), ("mask_stride", C.c_int64),
                ("z", C.c_void_p), ("ldz", C.c_int64), ("den", C.c_void_p), ("sw", C.c_void_p),
                ("nanflag", C.c_void_p),
                ("n_rows", C.c_int32), ("alpha", C.c_float),
                ("geom", AggGeom), ("hub", HubTasks)]


class AggBwdArgs(C.Structure):
    _fields_ = [("segptr", C.c_void_p), ("col", C.c_void_p), ("t1", C.c_void_p), ("t2", C.c_void_p),
                ("xrow", C.c_void_p), ("ldxr", C.c_int64), ("xcol", C.c_void_p), ("ldxc", C.c_int64),
                ("rel", C.c_void_p), ("ldr", C.c_int64),
                ("mask", C.c_void_p), ("mask_stride", C.c_int64),
                ("dz", C.c_void_p), ("ldz", C.c_int64),
                ("den", C.c_void_p), ("sw", C.c_void_p), ("dden", C.c_void_p),
                ("gx", C.c_void_p), ("ldgx", C.c_int64), ("gr", C.c_void_p), ("ldgr", C.c_int64),
                ("rowout", C.c_void_p), ("ldro", C.c_int64), ("rowsc", C.c_void_p), ("rec", C.c_void_p),
                ("n_rows", C.c_int32), ("alpha", C.c_float),
                ("geom", AggGeom), ("hub", HubTasks)]


_VP, _I64, _I32 = C.c_void_p, C.c_int64, C.c_int32

ALLOC_FN = C.CFUNCTYPE(C.c_void_p, C.c_void_p, C.c_int64)


class TripleGraphArgs(C.Structure):
    _fields_ = [("uptr", C.c_void_p), ("ut", C.c_void_p), ("ur0", C.c_void_p), ("ugs", C.c_void_p), ("uge", C.c_void_p),
                ("rs", C.c_void_p), ("n_nodes", C.c_int32), ("n_pairs", C.c_int32), ("n_triples", C.c_int32),
                ("reserved", C.c_int32)]


class NhopResult(C.Structure):
    _fields_ = [("adj_idx", C.c_void_p), ("adj_val", C.c_void_p), ("nhop", C.c_void_p), ("e1", C.c_int64), ("e2", C.c_int64)]


class LossBwdArgs(C.Structure):
    _fields_ = [("segptr", C.c_void_p), ("inc", C.c_void_p), ("coef", C.c_void_p), ("sgn", C.c_void_p),
                ("gscale", C.c_void_p), ("out", C.c_void_p), ("ldo", C.c_int64),
                ("n_seg", C.c_int32), ("width", C.c_int32), ("mode", C.c_int32), ("reserved", C.c_int32),
                ("hub", HubTasks)]


class SgdArgs(C.Structure):
    _fields_ = [("param", C.c_void_p * 16), ("grad", C.c_void_p * 16), ("numel", C.c_int64 * 16),
                ("count", C.c_int32), ("lr", C.c_float)]


# name -> (restype, argtypes); every symbol include/spkbgat.h declares
class AttnWeightsArgs(C.Structure):
    _fields_ = [("a", C.c_void_p * 4), ("a2", C.c_void_p * 4), ("da", C.c_void_p * 4), ("da2", C.c_void_p * 4),
                ("n_heads", C.c_int32), ("F", C.c_int32), ("Rd", C.c_int32), ("D", C.c_int32),
                ("mode", C.c_int32), ("d_pad", C.c_int32), ("width", C.c_int32),
                ("f_pad", C.c_int32), ("lz", C.c_int32), ("reserved", C.c_int32),
                ("W0", C.c_void_p), ("ld0", C.c_int64), ("W1", C.c_void_p), ("ld1", C.c_int64), ("W2", C.c_void_p)]


SIGNATURES = {
    "spk_abi_version": (_I32, []),
    "spk_last_error": (C.c_char_p, []),
    "spk_launch_count": (_I64, []),
    "spk_edges_concat": (_I32, [_VP, _I64, _VP, _VP, _I64, _VP, _VP, _VP, _VP, _I64, _I64, _VP, _VP]),
    "spk_pack_index_host": (_I32, [_VP, _I64, _I64, _I64, _I64, _VP, _I32]),
    "spk_iota_i32": (_I32, [_VP, _I64, _VP]),
    "spk_sort_workspace_bytes": (_I64, [_I64]),
    "spk_sort_pairs": (_I32, [_VP, _VP, _VP, _VP, _I64, _I32, _VP, C.POINTER(_I32), _VP]),
    "spk_segment_ptr": (_I32, [_VP, _I64, _I32, _VP, _VP]),
    "spk_gather_i32": (_I32, [_VP, _VP, _I64, _VP, _VP]),
    "spk_rel_incidence": (_I32, [_VP, _VP, _I64, _I32, _VP, _VP, _VP]),
    "spk_gemm_nn": (_I32, [_VP, _I64, _VP, _I64, _VP, _I64, _I64, _I32, _I32, _I32, _VP]),
    "spk_gemm_nn_tc_supported": (_I32, [_VP, _I64, _I64, _I32, _I32]),
    "spk_gemm_tc_workspace_floats": (_I64, [_I32, _I32]),
    "spk_gemm_nn_tc": (_I32, [_VP, _I64, _VP, _I64, _VP, _I64, _I64, _I32, _I32, _I32, _VP, _VP]),
    "spk_gemm_nn_tc_act": (_I32, [_VP, _I64, _VP, _I64, _VP, _I64, _I64, _I32, _I32, _I32, _I32, _VP, _VP]),
    "spk_elu_inplace": (_I32, [_VP, _I64, _I64, _I32, _VP]),
    "spk_agg_table": (_I32, [_VP, _I64, _VP, _VP, _I64, _I64, _I32, _I32, _VP]),
    "spk_agg_fwd": (_I32, [C.POINTER(AggFwdArgs), _VP]),
    "spk_agg_bwd_pre": (_I32, [_VP, _VP, _I64, _VP, _I32, _I32, _I32, _VP, _I64, _VP, _I64, _VP]),
    "spk_agg_bwd_rows": (_I32, [C.POINTER(AggBwdArgs), _VP]),
    "spk_agg_bwd_ctx": (_I32, [C.POINTER(AggBwdArgs), _VP]),
    "spk_agg_dx": (_I32, [_VP, _I64, _VP, _I64, _VP, _I64, _I32, _I32, _I32, _VP, _I64, _VP, _VP]),
    "spk_gemm_tn_tc_supported": (_I32, [_VP, _I64, _VP, _I64, _I64, _I32, _I32]),
    "spk_gemm_tn_tc_workspace_floats": (_I64, [_I64, _I32, _I32]),
    "spk_gemm_tn_tc": (_I32, [_VP, _I64, _VP, _I64, _VP, _I64, _I64, _I32, _I32, _I32, _VP, _VP]),
    "spk_gemm_tn_workspace_floats": (_I64, [_I64, _I32, _I32]),
    "spk_gemm_tn": (_I32, [_VP, _I64, _VP, _I64, _VP, _I64, _I64, _I32, _I32, _I32, _VP, _VP]),
    "spk_edge_attn_fwd": (_I32, [C.POINTER(EdgeFwdArgs), _VP]),
    "spk_edge_attn_bwd_rows": (_I32, [C.POINTER(EdgeBwdRowsArgs), _VP]),
    "spk_edge_attn_bwd_segments": (_I32, [C.POINTER(SegGatherArgs), _VP]),
    "spk_edge_attn_bwd_fused": (_I32, [C.POINTER(EdgeBwdFusedArgs), _VP]),
    "spk_edge_attn_bwd_split": (_I32, [C.POINTER(EdgeBwdSplitArgs), _VP]),
    "spk_spmm_rowsum_fwd": (_I32, [_VP, _VP, _VP, _I64, _I32, _VP, _I64, _I32, _VP]),
    "spk_spmm_rowsum_bwd": (_I32, [_VP, _VP, _I64, _I32, _VP, _I64, _I64, _VP]),
    "spk_rownorm": (_I32, [_VP, _I64, _VP, _I64, _I64, _I32, _VP]),
    "spk_residual_norm_fwd": (_I32, [_VP, _I64, _VP, _I64, _VP, _VP, _I64, _VP, _I64, _I32, _VP]),
    "spk_residual_norm_bwd": (_I32, [_VP, _I64, _VP, _I64, _VP, _VP, _VP, _I64, _VP, _I64, _I64, _I32, _VP]),
    "spk_mask_from_index": (_I32, [_VP, _I64, _VP, _I64, _VP, _VP]),
    "spk_attn_weights_fwd": (_I32, [_VP, _VP]),
    "spk_attn_weights_bwd": (_I32, [_VP, _VP]),
    "spk_inner_product_workspace_bytes": (_I64, []),
    "spk_inner_product": (_I32, [_VP, _VP, _I64, _VP, _VP, _I32, _VP]),
    "spk_margin_loss_partials": (_I64, [_I64]),
    "spk_margin_loss_fwd": (_I32, [_VP, _I64, _I64, _VP, _I64, _I64, _VP, _I64, _I64, _I32, C.c_float, _I32,
                                   _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "spk_triple_incidence": (_I32, [_VP, _I64, _I64, _I64, _VP, _VP, _VP, _VP, _VP, _VP]),
    "spk_margin_loss_bwd": (_I32, [C.POINTER(LossBwdArgs), _VP]),
    "spk_sgd_step": (_I32, [C.POINTER(SgdArgs), _VP]),
    "spk_triple_keys": (_I32, [_VP, _I64, _I64, _I64, _VP, _VP, _VP]),
    "spk_corrupt_triples": (_I32, [_VP, _I64, _I32, _VP, _I64, _I64, _I64, _VP, _VP, C.c_uint64, _VP, _VP, _VP]),
    "spk_nhop_build": (_I32, [C.POINTER(TripleGraphArgs), _VP, _I64, _I32, ALLOC_FN, _VP, C.POINTER(NhopResult), _VP]),
    "spk_gather_concat": (_I32, [_VP, _VP, _VP, _VP, _VP, _I32, _I64, _I32, _VP, _I64, _VP, _VP]),
    "spk_mlp_head_fwd": (_I32, [_VP, _I64, _VP, _VP, _VP, C.c_float, _I64, _I32, _VP, _VP]),
    "spk_mlp_head_bwd": (_I32, [_VP, _I64, _VP, _VP, C.c_float, _VP, _I64, _I32, _VP, _I64, _VP, _I64, _VP]),
    "spk_tanh_fwd": (_I32, [_VP, _I64, _I64, _I32, _VP]),
    "spk_tanh_bwd": (_I32, [_VP, _I64, _VP, _I64, _I64, _I32, _VP, _I64, _VP]),
    "spk_rank_scores": (_I32, [_VP, _I64, _VP, _I64, _VP, _VP, C.c_float, _I64, _I32, _I32, _VP, _I64, _VP]),
    "spk_linkpred_count": (_I32, [_VP, _I64, _I64, _VP, _I64, _I64, _VP, _VP, C.c_float, _I32, _VP, _VP, _I64, _I32,
                                  _VP, _I64, _VP, _VP, _VP, _VP, _VP]),
    "spk_linkpred_filter": (_I32, [_VP, _I64, _I64, _I64, _VP, C.c_float, _I32, _VP, _I64, _I32, _VP, _I64, _VP, _VP,
                                   _VP, _I64, _VP, _VP, _VP, _VP]),
    "spk_export_json": (_I32, [_VP, _I64, _I64, _I64, C.c_char_p, _I32]),
    "spk_export_bin": (_I32, [_VP, _I64, _I64, _I64, C.c_char_p]),
    "spk_import_json_shape": (_I32, [C.c_char_p, C.POINTER(_I64), C.POINTER(_I64)]),
    "spk_import_json": (_I32, [C.c_char_p, _VP, _I64, _I64, _I64, _I32]),
}

_lib = None
current_tag = ""          # optional label appended to the next timed call's name (see profiler.py)


class _Lib:
    """Thin proxy over the CDLL: identical calls; when `timing` is a list every kernel-launching entry
    point is bracketed by CUDA events on the launching stream (bench.py's per-kernel pass)."""

    def __init__(self, cdll):
        self._cdll = cdll
        self.timing = None

    def __getattr__(self, name):
        fn = getattr(self._cdll, name)
        if self.timing is None or SIGNATURES[name][1][-1:] != [_VP] or "workspace" in name or "supported" in name:
            return fn

        def timed(*args):
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = fn(*args)
            e1.record()
            global current_tag
            self.timing.append((name[4:] + (":" + current_tag if current_tag else ""), e0, e1))
            if "gemm" in name:
                current_tag = ""
            return rc
        return timed


def load():
    """Load libspkbgat.so, bind every declared symbol, check the ABI version. Raises if missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or make -C recon_b200/csrc). recon_b200 has no CPU / PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.spk_abi_version() != ABI_VERSION:
        raise RuntimeError(f"libspkbgat ABI {lib.spk_abi_version()} != binding {ABI_VERSION}")
    _lib = _Lib(lib)
    return _lib


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("recon_b200 ops need CUDA tensors (no CPU fallback)")
    return t.data_ptr()


def launch_count():
    """Kernels launched through libspkbgat so far (bench.py reports the delta as gpu_launches)."""
    return int(load().spk_launch_count())


def check(rc, what):
    if rc != 0:
        msg = load().spk_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libspkbgat {what} failed (code {rc}): {msg}")
