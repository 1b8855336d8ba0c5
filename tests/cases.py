"""Deterministic test-case factory shared by the golden generator, the oracle tests and the
GPU parity tests.

A case is described by a small JSON-able `spec`; parameters and inputs are regenerated from
`np.random.RandomState(seed)` (a frozen stream), so fixtures only need to store the spec, a
checksum of the regenerated inputs and the reference's outputs.

Parameter names are the reference's state-dict keys (SURVEY.md section 5, checkpoint row).
"""
from __future__ import annotations

import hashlib
import math
import os
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

from oracle import egnn_oracle as O  # noqa: E402  (tests are allowed to import the oracle)


# ------------------------------------------------------------------ parameter shapes


def layer_param_shapes(cfg):
    """Shapes of one EGNN layer's parameters (reference egnn_pytorch.py:178-208)."""
    E = O.edge_input_dim(cfg)
    d, m = cfg["dim"], cfg["m_dim"]
    shapes = {
        "edge_mlp.0.weight": (2 * E, E), "edge_mlp.0.bias": (2 * E,),
        "edge_mlp.3.weight": (m, 2 * E), "edge_mlp.3.bias": (m,),
    }
    if cfg["soft_edges"]:
        shapes.update({"edge_gate.0.weight": (1, m), "edge_gate.0.bias": (1,)})
    if cfg["norm_feats"]:
        shapes.update({"node_norm.weight": (d,), "node_norm.bias": (d,)})
    if cfg["norm_coors"]:
        shapes["coors_norm.scale"] = (1,)
    if cfg["update_feats"]:
        shapes.update({"node_mlp.0.weight": (2 * d, d + m), "node_mlp.0.bias": (2 * d,),
                       "node_mlp.3.weight": (d, 2 * d), "node_mlp.3.bias": (d,)})
    if cfg["update_coors"]:
        shapes.update({"coors_mlp.0.weight": (4 * m, m), "coors_mlp.0.bias": (4 * m,),
                       "coors_mlp.3.weight": (1, 4 * m), "coors_mlp.3.bias": (1,)})
    return shapes


def gen_layer_params(cfg, rs, init):
    """init='default': the reference's init (weights N(0, init_eps), biases PyTorch-default
    uniform, egnn_pytorch.py:217-222).  init='xavier': realistic-scale Xavier-normal weights,
    non-trivial LayerNorm affine and CoorsNorm scale (SURVEY.md section 4: the default init is
    bias-dominated and hides errors)."""
    out = {}
    for name, shp in layer_param_shapes(cfg).items():
        if name.endswith(".weight") and len(shp) == 2:
            fan_out, fan_in = shp
            std = cfg["init_eps"] if init == "default" else math.sqrt(2.0 / (fan_in + fan_out))
            out[name] = rs.standard_normal(shp) * std
        elif name.startswith("node_norm"):
            if init == "default":
                out[name] = np.ones(shp) if name.endswith("weight") else np.zeros(shp)
            else:
                base = 1.0 if name.endswith("weight") else 0.0
                out[name] = base + 0.2 * rs.standard_normal(shp)
        elif name == "coors_norm.scale":
            out[name] = np.full(shp, cfg["norm_coors_scale_init"] if init == "default" else 0.7)
        else:  # Linear bias
            wshape = layer_param_shapes(cfg)[name.replace(".bias", ".weight")]
            bound = 1.0 / math.sqrt(wshape[1])
            out[name] = rs.uniform(-bound, bound, shp)
    return out


def gen_network_params(ncfg, rs, init):
    out = {}
    d = ncfg["dim"]
    if ncfg["num_tokens"] is not None:
        out["token_emb.weight"] = rs.standard_normal((ncfg["num_tokens"], d))
    if ncfg["num_positions"] is not None:
        out["pos_emb.weight"] = rs.standard_normal((ncfg["num_positions"], d))
    if ncfg["num_edge_tokens"] is not None:
        out["edge_emb.weight"] = rs.standard_normal((ncfg["num_edge_tokens"], ncfg["edge_dim"]))
    if ncfg["num_adj_degrees"] is not None and ncfg["adj_dim"] > 0:
        out["adj_emb.weight"] = rs.standard_normal((ncfg["num_adj_degrees"] + 1, ncfg["adj_dim"]))
    for l in range(ncfg["depth"]):
        for k, v in gen_layer_params(ncfg["layer"], rs, init).items():
            out[f"layers.{l}.1.{k}"] = v
    # global linear attention blocks (reference egnn_pytorch.py:112-130), generated AFTER everything else so that the
    # parameter streams of the cases without them are unchanged
    if ncfg.get("global_layers"):
        inner = ncfg["global_heads"] * ncfg["global_dim_head"]
        out["global_tokens"] = rs.standard_normal((ncfg["num_global_tokens"], d))
        lin = lambda o, i: rs.standard_normal((o, i)) * math.sqrt(1.0 / i)
        for l in ncfg["global_layers"]:
            pre = f"layers.{l}.0."
            for nm in ("norm_seq", "norm_queries", "ff.0"):
                out[pre + nm + ".weight"] = 1.0 + 0.2 * rs.standard_normal((d,))
                out[pre + nm + ".bias"] = 0.1 * rs.standard_normal((d,))
            for a in ("attn1", "attn2"):
                out[pre + a + ".to_q.weight"] = lin(inner, d)
                out[pre + a + ".to_kv.weight"] = lin(2 * inner, d)
                out[pre + a + ".to_out.weight"] = lin(d, inner)
                out[pre + a + ".to_out.bias"] = 0.1 * rs.standard_normal((d,))
            out[pre + "ff.1.weight"] = lin(4 * d, d)
            out[pre + "ff.1.bias"] = 0.1 * rs.standard_normal((4 * d,))
            out[pre + "ff.3.weight"] = lin(d, 4 * d)
            out[pre + "ff.3.bias"] = 0.1 * rs.standard_normal((d,))
    return out


# ------------------------------------------------------------------ inputs


def chain_adjacency(n, diagonal=True):
    """README.md:89-90 style chain: adj[i,j] = |i-j| <= 1."""
    i = np.arange(n)
    a = np.abs(i[:, None] - i[None, :]) <= 1
    if not diagonal:
        a &= i[:, None] != i[None, :]
    return a


def gen_inputs(spec, rs):
    B, N, C = spec["B"], spec["N"], spec.get("C", 3)
    kind = spec["kind"]
    ins = {}
    if kind == "network":
        ncfg = spec["_ncfg"]
        d, edge_dim = ncfg["dim"], ncfg["edge_dim"]
        if ncfg["num_tokens"] is not None:
            ins["feats"] = rs.randint(0, ncfg["num_tokens"], (B, N))
        else:
            ins["feats"] = rs.standard_normal((B, N, d))
        if spec.get("edges", False):
            if ncfg["num_edge_tokens"] is not None:
                ins["edges"] = rs.randint(0, ncfg["num_edge_tokens"], (B, N, N))
            else:
                ins["edges"] = rs.standard_normal((B, N, N, edge_dim))
    else:
        cfg = spec["_cfg"]
        ins["feats"] = rs.standard_normal((B, N, cfg["dim"]))
        if cfg["edge_dim"] > 0:
            ins["edges"] = rs.standard_normal((B, N, N, cfg["edge_dim"]))
    ins["coors"] = rs.standard_normal((B, N, C)) * spec.get("coor_scale", 1.0)
    mk = spec.get("mask", "none")
    if mk == "full":
        ins["mask"] = np.ones((B, N), bool)
    elif mk == "padded":      # trailing padding, different length per graph
        lens = [max(2, N - 1 - (3 * b) % max(1, N // 3)) for b in range(B)]
        ins["mask"] = np.arange(N)[None, :] < np.asarray(lens)[:, None]
    elif mk == "random":
        m = rs.uniform(size=(B, N)) < 0.8
        m[:, :2] = True
        ins["mask"] = m
    elif mk == "one_empty":   # the last graph of the batch has no valid node at all
        m = np.ones((B, N), bool)
        m[-1] = False
        ins["mask"] = m
    adj = spec.get("adj", "none")
    if adj == "chain":
        ins["adj_mat"] = chain_adjacency(N, True)
    elif adj == "chain_nodiag":
        ins["adj_mat"] = chain_adjacency(N, False)
    elif adj == "random3d":   # batched, symmetric, sparse
        a = rs.uniform(size=(B, N, N)) < spec.get("adj_p", 0.15)
        a = a | a.transpose(0, 2, 1) | np.eye(N, dtype=bool)[None]   # keep the diagonal: see note below
        ins["adj_mat"] = a
    return ins


def build_case(spec):
    """spec -> dict(cfg|ncfg, params, inputs).  Deterministic in spec['seed']."""
    spec = dict(spec)
    rs = np.random.RandomState(spec["seed"])
    init = spec.get("init", "default")
    if spec["kind"] == "network":
        ncfg = O.network_cfg(**spec["cfg"])
        spec["_ncfg"] = ncfg
        params = gen_network_params(ncfg, rs, init)
        ins = gen_inputs(spec, rs)
        return dict(kind="network", ncfg=ncfg, params=params, inputs=ins, spec=spec)
    cfg = O.layer_cfg(**spec["cfg"])
    spec["_cfg"] = cfg
    params = gen_layer_params(cfg, rs, init)
    ins = gen_inputs(spec, rs)
    return dict(kind="layer", cfg=cfg, params=params, inputs=ins, spec=spec)


def case_checksum(case):
    """sha256 over the regenerated parameters and inputs (guards against RNG drift)."""
    h = hashlib.sha256()
    for group in (case["params"], case["inputs"]):
        for k in sorted(group):
            a = np.ascontiguousarray(group[k])
            h.update(k.encode())
            h.update(str(a.dtype).encode())
            h.update(a.tobytes())
    return h.hexdigest()


def run_oracle(case, dtype=np.float64, **kw):
    ins = case["inputs"]
    if case["kind"] == "network":
        return O.egnn_network_forward(case["params"], case["ncfg"], ins["feats"], ins["coors"],
                                      adj_mat=ins.get("adj_mat"), edges=ins.get("edges"),
                                      mask=ins.get("mask"), dtype=dtype, **kw)
    return O.egnn_layer_forward(case["params"], case["cfg"], ins["feats"], ins["coors"],
                                edges=ins.get("edges"), mask=ins.get("mask"),
                                adj_mat=ins.get("adj_mat"), dtype=dtype, **kw)


# ------------------------------------------------------------------ the case list
#
# Tie note: `torch.topk` does not define which of several equal-ranked candidates it keeps
# (SURVEY.md section 7.3 item 4).  Adjacent nodes all rank 0 (egnn_pytorch.py:256), so a case is
# only well-defined when k >= 1 + (number of adjacent nodes) for every row -- true whenever the
# adjacency carries its diagonal under `only_sparse_neighbors` (k = max row-sum, :249).  Cases
# that violate this are marked `tie_dependent` and are checked CUDA-vs-oracle only (both break
# ties towards the lowest index), never against the reference's outputs.

L = "layer"
NW = "network"

# Small cases exercising every EGNN kwarg (SURVEY.md section 4 "what these tests do not pin").
SPECS = {
    # --- dense all-pairs
    "dense_basic":        dict(kind=L, cfg=dict(dim=16), B=2, N=12, seed=1),
    "dense_xavier":       dict(kind=L, cfg=dict(dim=32), B=2, N=20, seed=2, init="xavier"),
    "dense_edges":        dict(kind=L, cfg=dict(dim=16, edge_dim=4), B=2, N=10, seed=3, init="xavier"),
    "dense_mask_padded":  dict(kind=L, cfg=dict(dim=16, edge_dim=2), B=3, N=14, seed=4, init="xavier", mask="padded"),
    "dense_mask_random":  dict(kind=L, cfg=dict(dim=8), B=2, N=17, seed=5, init="xavier", mask="random"),
    "dense_soft_edges":   dict(kind=L, cfg=dict(dim=16, soft_edges=True), B=1, N=9, seed=6, init="xavier"),
    "dense_norm_coors":   dict(kind=L, cfg=dict(dim=16, norm_coors=True), B=2, N=11, seed=7, init="xavier"),
    "dense_clamp":        dict(kind=L, cfg=dict(dim=16, coor_weights_clamp_value=0.05), B=2, N=13, seed=8, init="xavier", mask="padded"),
    "dense_mean":         dict(kind=L, cfg=dict(dim=16, m_pool_method="mean"), B=2, N=10, seed=9, init="xavier"),
    "dense_mean_masked":  dict(kind=L, cfg=dict(dim=16, m_pool_method="mean"), B=3, N=10, seed=10, init="xavier", mask="padded"),
    "dense_fourier":      dict(kind=L, cfg=dict(dim=8, fourier_features=3, edge_dim=2), B=2, N=9, seed=11, init="xavier"),
    "dense_c5":           dict(kind=L, cfg=dict(dim=16, edge_dim=4), B=1, N=8, C=5, seed=12, init="xavier", mask="full"),
    "dense_c2":           dict(kind=L, cfg=dict(dim=8), B=2, N=7, C=2, seed=13, init="xavier"),
    "dense_norm_feats":   dict(kind=L, cfg=dict(dim=24, norm_feats=True), B=2, N=9, seed=14, init="xavier"),
    "dense_no_feats":     dict(kind=L, cfg=dict(dim=16, update_feats=False), B=2, N=9, seed=15, init="xavier"),
    "dense_no_coors":     dict(kind=L, cfg=dict(dim=16, update_coors=False), B=2, N=9, seed=16, init="xavier"),
    "dense_mdim8":        dict(kind=L, cfg=dict(dim=16, m_dim=8), B=2, N=9, seed=17, init="xavier"),
    "dense_mdim32":       dict(kind=L, cfg=dict(dim=12, m_dim=32, edge_dim=1), B=1, N=9, seed=18, init="xavier"),
    "dense_everything":   dict(kind=L, cfg=dict(dim=20, edge_dim=3, fourier_features=2, norm_feats=True, norm_coors=True,
                                              soft_edges=True, coor_weights_clamp_value=1.5, m_pool_method="mean"),
                               B=2, N=15, seed=19, init="xavier", mask="padded"),
    # BASELINE config c1: EGNN(dim=512), B=1, N=16
    "c1_dim512":          dict(kind=L, cfg=dict(dim=512), B=1, N=16, seed=20),
    "c1_dim512_xavier":   dict(kind=L, cfg=dict(dim=512, edge_dim=4), B=1, N=16, seed=21, init="xavier", mask="full"),
    # --- k nearest neighbours
    "knn_basic":          dict(kind=L, cfg=dict(dim=16, num_nearest_neighbors=4), B=2, N=20, seed=30, init="xavier"),
    "knn_edges_mask":     dict(kind=L, cfg=dict(dim=16, edge_dim=3, num_nearest_neighbors=5), B=3, N=18, seed=31, init="xavier", mask="padded"),
    "knn_radius_mask":    dict(kind=L, cfg=dict(dim=16, num_nearest_neighbors=6, valid_radius=1.5), B=2, N=24, seed=32, init="xavier", mask="full"),
    "knn_radius_nomask":  dict(kind=L, cfg=dict(dim=16, num_nearest_neighbors=6, valid_radius=1.5), B=2, N=24, seed=33, init="xavier"),
    "knn_norm_coors":     dict(kind=L, cfg=dict(dim=16, edge_dim=1, num_nearest_neighbors=8, norm_coors=True), B=1, N=40, seed=34, init="xavier", mask="full"),
    "knn_mean_fourier":   dict(kind=L, cfg=dict(dim=8, num_nearest_neighbors=7, m_pool_method="mean", fourier_features=2), B=2, N=21, seed=35, init="xavier", mask="random"),
    "knn_k_eq_n":         dict(kind=L, cfg=dict(dim=8, num_nearest_neighbors=9), B=2, N=9, seed=36, init="xavier"),
    "knn_k33":            dict(kind=L, cfg=dict(dim=8, num_nearest_neighbors=33), B=1, N=70, seed=37, init="xavier", mask="padded"),
    "knn_k32_c5":         dict(kind=L, cfg=dict(dim=8, num_nearest_neighbors=32, edge_dim=2), B=1, N=50, C=5, seed=38, init="xavier"),
    # --- adjacency
    "adj_knn_chain":      dict(kind=L, cfg=dict(dim=16, num_nearest_neighbors=5), B=2, N=16, seed=40, init="xavier", adj="chain", mask="padded"),
    "adj_sparse_chain":   dict(kind=L, cfg=dict(dim=16, only_sparse_neighbors=True), B=2, N=16, seed=41, init="xavier", adj="chain", mask="full"),
    "adj_sparse_nomask":  dict(kind=L, cfg=dict(dim=16, only_sparse_neighbors=True), B=2, N=16, seed=42, init="xavier", adj="chain"),
    "adj_sparse_random":  dict(kind=L, cfg=dict(dim=12, edge_dim=2, only_sparse_neighbors=True), B=2, N=20, seed=43, init="xavier", adj="random3d", mask="padded"),
    "adj_sparse_nodiag":  dict(kind=L, cfg=dict(dim=12, only_sparse_neighbors=True, num_nearest_neighbors=3), B=1, N=12, seed=44, init="xavier", adj="chain_nodiag", mask="full",
                               tie_dependent=True),   # k=2 < {self, i-1, i+1}: torch.topk's tie order decides
    # --- network
    "net_c3_small":       dict(kind=NW, cfg=dict(depth=3, dim=32, num_tokens=21, num_positions=64, num_nearest_neighbors=8,
                                                 coor_weights_clamp_value=2.0), B=1, N=48, seed=50, mask="full"),
    "net_c3_xavier":      dict(kind=NW, cfg=dict(depth=2, dim=16, num_tokens=21, num_positions=40, num_nearest_neighbors=6,
                                                 coor_weights_clamp_value=2.0), B=2, N=30, seed=51, init="xavier", mask="padded"),
    "net_dense_feats":    dict(kind=NW, cfg=dict(depth=2, dim=16, edge_dim=3), B=2, N=10, seed=52, init="xavier", edges=True),
    "net_edge_tokens":    dict(kind=NW, cfg=dict(depth=2, dim=16, num_tokens=11, num_edge_tokens=5, edge_dim=4,
                                                 num_nearest_neighbors=3), B=2, N=12, seed=53, init="xavier", edges=True, mask="full"),
    "net_adj_degrees":    dict(kind=NW, cfg=dict(depth=2, dim=16, num_tokens=21, num_adj_degrees=2, adj_dim=4,
                                                 num_nearest_neighbors=6), B=2, N=14, seed=54, init="xavier", adj="chain", mask="padded"),
    "net_c5_small":       dict(kind=NW, cfg=dict(depth=3, dim=32, num_tokens=21, num_adj_degrees=3, adj_dim=8,
                                                 only_sparse_neighbors=True), B=1, N=40, seed=55, adj="chain", mask="full"),
    "net_c5_xavier":      dict(kind=NW, cfg=dict(depth=2, dim=16, num_tokens=21, num_adj_degrees=3, adj_dim=8,
                                                 only_sparse_neighbors=True, edge_dim=2), B=2, N=24, seed=56, init="xavier",
                               adj="chain", mask="padded", edges=True),
    "net_adj_dense":      dict(kind=NW, cfg=dict(depth=2, dim=12, num_tokens=9, num_adj_degrees=2, adj_dim=3), B=2, N=11, seed=58,
                               init="xavier", adj="chain", mask="padded"),   # degree labels on DENSE layers (no neighbour selection)
    "net_adj_random":     dict(kind=NW, cfg=dict(depth=2, dim=12, num_adj_degrees=2, adj_dim=3, only_sparse_neighbors=True),
                               B=2, N=16, seed=57, init="xavier", adj="random3d", adj_p=0.1, mask="full"),
    # EGNN_Network with GlobalLinearAttention blocks (reference egnn_pytorch.py:81-144, :381-385, :439-446)
    "net_global_attn":    dict(kind=NW, cfg=dict(depth=2, dim=16, num_tokens=9, global_linear_attn_every=1, global_linear_attn_heads=2,
                                                 global_linear_attn_dim_head=8, num_global_tokens=3), B=2, N=14, seed=59,
                               init="xavier", mask="padded"),
    "net_global_every2":  dict(kind=NW, cfg=dict(depth=3, dim=24, global_linear_attn_every=2, global_linear_attn_heads=4,
                                                 global_linear_attn_dim_head=16, num_global_tokens=4, num_nearest_neighbors=5,
                                                 norm_coors=True), B=2, N=20, seed=60, init="xavier"),
    "net_global_allmask": dict(kind=NW, cfg=dict(depth=1, dim=16, global_linear_attn_every=1, global_linear_attn_heads=2,
                                                 global_linear_attn_dim_head=8, num_global_tokens=2), B=2, N=9, seed=61,
                               init="xavier", mask="one_empty"),     # one graph fully masked: uniform attention (:101-104)
}


# ------------------------------------------------------------------ gradients (backward parity)
#
# Loss = sum(feats_out * G_f) + sum(coors_out * G_x) with fixed random cotangents G_f, G_x, so one
# backward pass exercises every output element.  The huge-parameter c1 cases are left out of the committed
# gradient fixtures (25 MB each in float64); they are still checked CUDA-vs-oracle.

# (the global-attention blocks train through PyTorch autograd, not through egnn_layer_backward: no hand-written gradient)
# knn_k33 / knn_k32_c5 have no committed reference-gradient fixture; tests/test_gpu_grad_shapes.py checks their
# gradients against the numpy oracle.
GRAD_SPECS = [n for n in SPECS if not n.startswith("c1_") and not n.startswith("net_global") and n not in {"knn_k33", "knn_k32_c5"}]


def upstream_grads(case):
    """Deterministic cotangents for (feats_out, coors_out)."""
    spec = case["spec"]
    rs = np.random.RandomState(spec["seed"] + 100003)
    B, N, C = spec["B"], spec["N"], spec.get("C", 3)
    d = case["ncfg"]["dim"] if case["kind"] == "network" else case["cfg"]["dim"]
    return rs.standard_normal((B, N, d)), rs.standard_normal((B, N, C))


def run_oracle_grad(case):
    """-> dict(feats|None, coors, edges|None, params{key: grad}) from the numpy backward oracle."""
    from oracle import egnn_oracle_grad as G
    ins = case["inputs"]
    gf, gx = upstream_grads(case)
    if case["kind"] == "network":
        return G.egnn_network_backward(case["params"], case["ncfg"], ins["feats"], ins["coors"], ins.get("adj_mat"),
                                       ins.get("edges"), ins.get("mask"), gf, gx)
    return G.egnn_layer_backward(case["params"], case["cfg"], ins["feats"], ins["coors"], ins.get("edges"),
                                 ins.get("mask"), ins.get("adj_mat"), gf, gx)


def flatten_grads(r):
    """dict from run_oracle_grad / the fixtures -> flat {name: array} ('in.feats', 'in.coors', 'in.edges', 'p.<key>')."""
    out = {}
    for k in ("feats", "coors", "edges"):
        if r.get(k) is not None:
            out[f"in.{k}"] = np.asarray(r[k])
    for k, v in r["params"].items():
        out[f"p.{k}"] = np.asarray(v)
    return out
