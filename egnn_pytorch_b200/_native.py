"""ctypes binding of libegnn_b200.so (the C ABI declared in include/egnn_b200.h).

There is no CPU fallback: if the shared library is missing or does not export the expected
symbols, importing the kernels fails loudly.  Build it with `python -m egnn_pytorch_b200.build`
(or `__graft_entry__.build()`); it is compiled for sm_100a only.
"""
from __future__ import annotations

import ctypes as C
import os

ABI_VERSION = 3

DTYPE_F32, DTYPE_F64, DTYPE_BF16 = 0, 1, 2

FLAG_NORM_FEATS = 1 << 0
FLAG_NORM_COORS = 1 << 1
FLAG_UPDATE_FEATS = 1 << 2
FLAG_UPDATE_COORS = 1 << 3
FLAG_SOFT_EDGES = 1 << 4
FLAG_POOL_MEAN = 1 << 5
FLAG_CLAMP = 1 << 6
FLAG_ONLY_SPARSE = 1 << 7
FLAG_ADJ_BATCHED = 1 << 8

ERR_UNSUPPORTED = -3

LIB_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib")
LIB_PATH = os.environ.get("EGNN_B200_LIB") or os.path.join(LIB_DIR, "libegnn_b200.so")   # override: A/B runs of kernel variants


class LayerDesc(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("dtype", C.c_int32), ("B", C.c_int32), ("N", C.c_int32),
        ("C", C.c_int32), ("dim", C.c_int32), ("edge_dim", C.c_int32), ("label_dim", C.c_int32),
        ("num_labels", C.c_int32), ("m_dim", C.c_int32), ("fourier", C.c_int32), ("k", C.c_int32),
        ("flags", C.c_uint32), ("row_begin", C.c_int32), ("row_end", C.c_int32), ("reserved", C.c_int32),
        ("valid_radius", C.c_double), ("clamp", C.c_double), ("dropout_p", C.c_double), ("dropout_seed", C.c_uint64),
    ]


WEIGHT_FIELDS = (
    "edge_w1", "edge_b1", "edge_w2", "edge_b2", "gate_w", "gate_b", "norm_g", "norm_b", "coors_scale",
    "node_w1", "node_b1", "node_w2", "node_b2", "coors_w1", "coors_b1", "coors_w2", "coors_b2", "label_emb",
)

# state-dict key (reference naming, SURVEY.md section 5) -> EgnnLayerWeights field
STATE_KEY_TO_FIELD = {
    "edge_mlp.0.weight": "edge_w1", "edge_mlp.0.bias": "edge_b1",
    "edge_mlp.3.weight": "edge_w2", "edge_mlp.3.bias": "edge_b2",
    "edge_gate.0.weight": "gate_w", "edge_gate.0.bias": "gate_b",
    "node_norm.weight": "norm_g", "node_norm.bias": "norm_b",
    "coors_norm.scale": "coors_scale",
    "node_mlp.0.weight": "node_w1", "node_mlp.0.bias": "node_b1",
    "node_mlp.3.weight": "node_w2", "node_mlp.3.bias": "node_b2",
    "coors_mlp.0.weight": "coors_w1", "coors_mlp.0.bias": "coors_b1",
    "coors_mlp.3.weight": "coors_w2", "coors_mlp.3.bias": "coors_b2",
}


class LayerWeights(C.Structure):
    _fields_ = [(name, C.c_void_p) for name in WEIGHT_FIELDS]


class LayerIO(C.Structure):
    _fields_ = [
        ("feats", C.c_void_p), ("coors", C.c_void_p), ("edges", C.c_void_p), ("edge_labels", C.c_void_p),
        ("mask", C.c_void_p), ("adj", C.c_void_p), ("feats_out", C.c_void_p), ("coors_out", C.c_void_p),
        ("nbr_idx", C.c_void_p), ("pre2_out", C.c_void_p),
    ]


class LayerWeightGrads(C.Structure):
    _fields_ = [(name, C.c_void_p) for name in WEIGHT_FIELDS]


class LayerGrads(C.Structure):
    _fields_ = [("g_feats_out", C.c_void_p), ("g_coors_out", C.c_void_p), ("g_feats", C.c_void_p),
                ("g_coors", C.c_void_p), ("g_edges", C.c_void_p), ("w", LayerWeightGrads)]


GA_WEIGHT_FIELDS = ("norm_seq_g", "norm_seq_b", "norm_q_g", "norm_q_b", "a1_wq", "a1_wkv", "a1_wo", "a1_bo", "a2_wq", "a2_wkv", "a2_wo",
                    "a2_bo", "ff_ln_g", "ff_ln_b", "ff_w1", "ff_b1", "ff_w2", "ff_b2")
# GlobalLinearAttention state-dict key (reference naming) -> EgnnGlobalAttnWeights field
GA_STATE_KEY_TO_FIELD = {
    "norm_seq.weight": "norm_seq_g", "norm_seq.bias": "norm_seq_b", "norm_queries.weight": "norm_q_g", "norm_queries.bias": "norm_q_b",
    "attn1.to_q.weight": "a1_wq", "attn1.to_kv.weight": "a1_wkv", "attn1.to_out.weight": "a1_wo", "attn1.to_out.bias": "a1_bo",
    "attn2.to_q.weight": "a2_wq", "attn2.to_kv.weight": "a2_wkv", "attn2.to_out.weight": "a2_wo", "attn2.to_out.bias": "a2_bo",
    "ff.0.weight": "ff_ln_g", "ff.0.bias": "ff_ln_b", "ff.1.weight": "ff_w1", "ff.1.bias": "ff_b1", "ff.3.weight": "ff_w2", "ff.3.bias": "ff_b2",
}


class GlobalAttnDesc(C.Structure):
    _fields_ = [("abi_version", C.c_int32), ("dtype", C.c_int32), ("B", C.c_int32), ("N", C.c_int32), ("T", C.c_int32),
                ("dim", C.c_int32), ("heads", C.c_int32), ("dim_head", C.c_int32)]


class GlobalAttnWeights(C.Structure):
    _fields_ = [(name, C.c_void_p) for name in GA_WEIGHT_FIELDS]


class GlobalAttnIO(C.Structure):
    _fields_ = [("x", C.c_void_p), ("queries", C.c_void_p), ("mask", C.c_void_p), ("x_out", C.c_void_p), ("queries_out", C.c_void_p)]


# every symbol include/egnn_b200.h declares: (restype, argtypes)
_P = C.POINTER
SYMBOLS = {
    "egnn_abi_version": (C.c_int, []),
    "egnn_strerror": (C.c_char_p, [C.c_int]),
    "egnn_layer_packed_bytes": (C.c_int, [_P(LayerDesc), _P(C.c_size_t)]),
    "egnn_layer_pack_weights": (C.c_int, [_P(LayerDesc), _P(LayerWeights), C.c_void_p, C.c_size_t, C.c_void_p]),
    "egnn_layer_workspace_bytes": (C.c_int, [_P(LayerDesc), _P(C.c_size_t)]),
    "egnn_layer_forward": (C.c_int, [_P(LayerDesc), _P(LayerWeights), C.c_void_p, _P(LayerIO), C.c_void_p,
                                     C.c_size_t, C.c_void_p]),
    "egnn_layer_forward_host": (C.c_int, [_P(LayerDesc), _P(LayerWeights), C.c_void_p, _P(LayerIO), C.c_void_p]),
    "egnn_layer_backward_workspace_bytes": (C.c_int, [_P(LayerDesc), _P(C.c_size_t)]),
    "egnn_layer_backward": (C.c_int, [_P(LayerDesc), _P(LayerWeights), C.c_void_p, _P(LayerIO), C.c_void_p,
                                      _P(LayerGrads), C.c_void_p, C.c_size_t, C.c_void_p]),
    "egnn_knn_select": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_int32, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]),
    "egnn_adj_neighbors": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "egnn_adj_workspace_bytes": (C.c_int, [C.c_int32, C.c_int32, _P(C.c_size_t)]),
    "egnn_adj_expand": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "egnn_embed_nodes": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p]),
    "egnn_gemm_bf16": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_int32,
                                 C.c_void_p, C.c_int32, C.c_void_p]),
    "egnn_global_attn_workspace_bytes": (C.c_int, [C.POINTER(GlobalAttnDesc), C.POINTER(C.c_size_t)]),
    "egnn_global_attn_forward": (C.c_int, [C.POINTER(GlobalAttnDesc), C.POINTER(GlobalAttnWeights), C.POINTER(GlobalAttnIO), C.c_void_p,
                                           C.c_size_t, C.c_void_p]),
    "egnn_comm_create": (C.c_int, [C.c_int32, C.c_int32, C.c_size_t, _P(C.c_void_p), C.c_void_p]),
    "egnn_comm_connect": (C.c_int, [C.c_void_p, C.c_void_p]),
    "egnn_comm_allgather": (C.c_int, [C.c_void_p, C.c_int32, _P(C.c_void_p), _P(C.c_size_t), _P(C.c_size_t), _P(C.c_void_p),
                                      C.c_void_p]),
    "egnn_comm_status": (C.c_int, [C.c_void_p, _P(C.c_int32)]),
    "egnn_comm_destroy": (C.c_int, [C.c_void_p]),
    "egnn_profile_enable": (C.c_int, [C.c_int]),
    "egnn_profile_read": (C.c_int, [_P(C.c_float), _P(C.c_int32), _P(C.c_int64), C.c_int]),
}

_lib = None


class NativeLibraryError(RuntimeError):
    pass


def load():
    """dlopen the library once and type every entry point."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryError(
            f"{LIB_PATH} not found: egnn_pytorch_b200 has no CPU fallback. Build the sm_100a library with "
            f"`python -m egnn_pytorch_b200.build` (needs nvcc).")
    try:
        lib = C.CDLL(LIB_PATH)
    except OSError as e:  # pragma: no cover
        raise NativeLibraryError(f"cannot load {LIB_PATH}: {e}") from e
    for name, (res, args) in SYMBOLS.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise NativeLibraryError(f"{LIB_PATH} does not export {name}; rebuild it") from e
        fn.restype = res
        fn.argtypes = args
    if lib.egnn_abi_version() != ABI_VERSION:
        raise NativeLibraryError(f"ABI mismatch: library {lib.egnn_abi_version()} vs binding {ABI_VERSION}")
    _lib = lib
    return lib


def strerror(code: int) -> str:
    return load().egnn_strerror(code).decode()


class EgnnNativeError(RuntimeError):
    def __init__(self, fn, code, detail=None):
        self.code = code
        super().__init__(f"{fn} failed: {strerror(code)} (code {code})" + (f": {detail}" if detail else ""))


def check(fn: str, code: int):
    if code != 0:
        raise EgnnNativeError(fn, code)
