"""ctypes binding of ``libxpgnn_b200.so`` (the C ABI declared in ``include/xpgnn_b200.h``).

The product path has no fallback: if the shared library is missing or a call fails, an
exception is raised.  Build it with ``python -m bikg_graph_explainability_public_b200.build``
(or ``__graft_entry__.build()``).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libxpgnn_b200.so")

i32, i64, u32, f32, f64 = C.c_int32, C.c_int64, C.c_uint32, C.c_float, C.c_double
ptr = C.c_void_p


class MaskPlan(C.Structure):
    _fields_ = [("n_elements", i32), ("n_communities", i32), ("n_positions", i32), ("n_rows", i32),
                ("com_ptr", ptr), ("com_idx", ptr), ("node_ptr", ptr), ("node_com", ptr),
                ("node_slot", ptr), ("order", ptr), ("size", ptr), ("size_int", ptr), ("row_start", ptr)]


class Relation(C.Structure):
    _fields_ = [("conv_kind", i32), ("src_lo", i32), ("src_hi", i32), ("dst_lo", i32), ("dst_hi", i32),
                ("n_edges", i32), ("rowptr", ptr), ("col", ptr), ("w_nbr", ptr), ("b_nbr", ptr), ("w_root", ptr)]


class Layer(C.Structure):
    _fields_ = [("n_rel", i32), ("rel_host", C.POINTER(Relation)), ("h_in", i32), ("h_out", i32), ("act", i32)]


class Dense(C.Structure):
    _fields_ = [("in_", i32), ("out", i32), ("act", i32), ("w", ptr), ("b", ptr)]


class Plan(C.Structure):
    _fields_ = [("n_nodes", i32), ("f_in", i32), ("x", ptr), ("n_layers", i32), ("layers_host", C.POINTER(Layer)),
                ("n_head", i32), ("head_host", C.POINTER(Dense)), ("n_query", i32), ("query", ptr),
                ("out_col", i32), ("prune", i32), ("hop", ptr), ("zero_edge_rule", i32), ("precision", i32)]


class FitQuery(C.Structure):
    _fields_ = [("act_off", i64), ("y_off", i64), ("kern_off", i64), ("w_off", i64), ("n", i32), ("s", i32), ("batch", i32),
                ("pad_", i32), ("losses", ptr)]


CONV_GCN, CONV_SAGE_MEAN = 0, 1
ACT_NONE, ACT_RELU, ACT_SIGMOID = 0, 1, 2

_SIGNATURES = {
    "xpgnn_last_error": (C.c_char_p, []),
    "xpgnn_abi_version": (C.c_int, []),
    "xpgnn_launch_count": (i64, []),
    "xpgnn_set_option": (C.c_int, [C.c_char_p, i32]),
    "xpgnn_get_option": (C.c_int, [C.c_char_p, C.POINTER(i32)]),
    "xpgnn_mt19937_draw": (C.c_int, [ptr, ptr, ptr, i64, ptr]),
    "xpgnn_mask_max_draws": (i64, [ptr, ptr, ptr, i32, i32, i32]),
    "xpgnn_mask_resolve": (C.c_int, [C.POINTER(MaskPlan), ptr, ptr, ptr, i32, ptr, ptr]),
    "xpgnn_mask_expand": (C.c_int, [C.POINTER(MaskPlan), ptr, ptr, ptr, i32, ptr, ptr, i32, ptr, ptr, ptr]),
    "xpgnn_shapley_expand": (C.c_int, [ptr, ptr, i32, i32, ptr, ptr, i32, ptr, ptr]),
    "xpgnn_randperm": (C.c_int, [ptr, i32, ptr, ptr]),
    "xpgnn_pack_mask": (C.c_int, [ptr, i32, i32, ptr, i32, ptr, ptr]),
    "xpgnn_khop_subgraph": (C.c_int, [ptr, i64, i64, i64, i32, ptr, ptr, ptr, ptr, ptr, ptr, ptr]),
    "xpgnn_build_csr": (C.c_int, [ptr, ptr, i64, i64, i32, ptr, ptr, ptr, ptr]),
    "xpgnn_khop_multi_workspace_bytes": (i64, [i64, i32]),
    "xpgnn_khop_multi_count": (C.c_int, [ptr, i64, i64, ptr, i32, i32, ptr, i64, ptr, ptr]),
    "xpgnn_khop_multi_emit": (C.c_int, [ptr, i64, i64, ptr, i32, i32, ptr, i64, ptr, ptr, ptr, i64, ptr, ptr, ptr, ptr, ptr,
                                        ptr]),
    "xpgnn_forward_workspace_bytes": (i64, [C.POINTER(Plan), i32]),
    "xpgnn_forward": (C.c_int, [C.POINTER(Plan), ptr, i32, i32, i32, ptr, ptr, i64, ptr, ptr]),
    "xpgnn_dense_rows": (C.c_int, [ptr, i64, i32, i32, ptr, ptr, i32, i32, ptr, i32, i32, i32, ptr]),
    "xpgnn_profile": (C.c_int, [i32]),
    "xpgnn_profile_read": (C.c_int, [ptr, ptr]),
    "xpgnn_shap_weights": (C.c_int, [ptr, i32, i32, i32, ptr, ptr, i32, ptr, ptr]),
    "xpgnn_wlm_fit": (C.c_int, [ptr, i32, i32, i32, i32, ptr, ptr, ptr, f64, f64, f64, i32, ptr, ptr]),
    "xpgnn_wlm_fit_batch": (C.c_int, [ptr, i32, ptr, i64, ptr, ptr, C.POINTER(FitQuery), i32, f64, f64, f64, i32, ptr]),
    "xpgnn_repeat_stats": (C.c_int, [ptr, i32, i32, ptr, ptr, ptr]),
    "xpgnn_community_mean": (C.c_int, [ptr, ptr, ptr, i32, ptr, ptr]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)
_lib = None


class XpgnnError(RuntimeError):
    pass


def load():
    """Load the shared library (no GPU needed for loading or symbol lookup)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise XpgnnError(
            "libxpgnn_b200.so is not built (%s). Run `python -m bikg_graph_explainability_public_b200.build`; "
            "there is no CPU fallback for the perturbation path." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.xpgnn_abi_version() != 1:
        raise XpgnnError("ABI version mismatch")
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise XpgnnError(load().xpgnn_last_error().decode())


def dptr(t):
    """Device pointer of a tensor (or NULL)."""
    return None if t is None else t.data_ptr()


def stream_ptr():
    import torch

    return torch.cuda.current_stream().cuda_stream


def set_options(**kv):
    """Engine options (``xpgnn_set_option``); returns the previous values."""
    lib, old = load(), {}
    for k, v in kv.items():
        prev = i32(0)
        check(lib.xpgnn_get_option(k.encode(), C.byref(prev)))
        old[k] = prev.value
        check(lib.xpgnn_set_option(k.encode(), int(v)))
    return old


def launch_count():
    return int(load().xpgnn_launch_count())
