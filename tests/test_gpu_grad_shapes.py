"""The SIMT forward and the hand-written backward at the shapes where their kernels tile.

The cases of `cases.SPECS` are small (N <= 70, dim <= 32 outside c1), so most of the tiling of the fp32 / fp64 kernels
never happens there: several row blocks of `pair_bwd2_dense_kernel`, more than one 128-channel block, k > 32 slots in
`pair_bwd2_knn_kernel`, the generic Q loop, split-K `dW` GEMMs, more than one row block in `colsum_acc_kernel`, the
GEMM routes of the per-node stages, the thread-per-pair dense fallback.  Each case below is sized to force one of those
(the `forces` note), and is checked against the numpy oracles (`oracle/`) in fp64 and fp32, forward and gradients,
with the per-pair pre-activations saved by the forward and recomputed by the backward.

`test_kernel_instantiations_are_exercised` fails when a dispatch change moves a case off the kernel it was written
for.  The preflight tests check that `egnn_layer_backward_workspace_bytes` accepts exactly the configurations the
backward kernels can launch, so an unsupported one fails at the forward call instead of at `loss.backward()`."""
import ctypes as C
import functools
import re

import numpy as np
import pytest
import torch

import cases
import util
from oracle import egnn_oracle as O
from oracle import egnn_oracle_grad as G

L, NW = "layer", "network"
F64, F32 = torch.float64, torch.float32
BOTH = (F64, F32)


def _edge_list(B, N, k, seed):
    """Random duplicate-free lists with empty (-1) slots: every third node has three empty slots, one node has none."""
    rs = np.random.RandomState(seed)
    nb = np.stack([np.stack([rs.permutation(N)[:k] for _ in range(N)]) for _ in range(B)]).astype(np.int64)
    nb[:, ::3, -3:] = -1
    nb[0, 5, :] = -1
    return nb


# name: spec (cases.build_case), grads = dtypes whose gradients are checked, and what the case forces
SHAPES = {
    # Hp = 296: three channel blocks, the last partial; 4 bwd2 row blocks (the last has 1 row); Q = 4 (generic loop);
    # dim > 64: tables and node update through launch_gemm; M = 194: split-K dW and 4 colsum row blocks
    "dense_tail_gemm": dict(spec=dict(kind=L, cfg=dict(dim=72, edge_dim=3), B=2, N=97, seed=401, init="xavier", mask="padded"),
                            grads=BOTH),
    # SIMPLE dense bwd2 (Q = 1) with a 6-row tail block; Hp = 168 = 128 + 40; mean pooling under a mask
    "dense_simple_all": dict(spec=dict(kind=L, cfg=dict(dim=40, soft_edges=True, norm_coors=True, coor_weights_clamp_value=0.3,
                                                        m_pool_method="mean"), B=3, N=70, seed=402, init="xavier", mask="random"),
                             grads=BOTH),
    # fourier chain in bwd3, C = 5, a 1-row tail block
    "dense_fourier_c5": dict(spec=dict(kind=L, cfg=dict(dim=32, fourier_features=2, edge_dim=2), B=2, N=33, C=5, seed=403,
                                       init="xavier"), grads=BOTH),
    # MP = 32 dense bwd1 / bwd2 over two row blocks (fp64 with m_dim = 32 is not trainable: see the preflight tests)
    "dense_mdim32": dict(spec=dict(kind=L, cfg=dict(dim=24, m_dim=32, edge_dim=2), B=2, N=45, seed=404, init="xavier"),
                         grads=(F32,)),
    # degree-label table (NL = 4) in dense bwd2 over three row blocks (CoorsNorm and xavier weights scaled by 0.5 keep
    # the second layer's distances O(10): plain xavier sends them to 1e4 over 70 neighbours)
    "net_dense_labels": dict(spec=dict(kind=NW, cfg=dict(depth=2, dim=24, num_adj_degrees=3, adj_dim=4, norm_coors=True), B=2,
                                       N=70, seed=405, init="xavier", adj="chain", mask="padded"), grads=BOTH, weight_scale=0.5),
    # both sides of simt_hsplit: B*N^2 = 4096 (two-phase dense kernel) and 4225 (one phase)
    "c1_hsplit_n64": dict(spec=dict(kind=L, cfg=dict(dim=512), B=1, N=64, seed=406, init="xavier"), grads=BOTH),
    "c1_hsplit_n65": dict(spec=dict(kind=L, cfg=dict(dim=512), B=1, N=65, seed=407, init="xavier"), grads=BOTH),
    # k = 33: two slot steps per row in bwd2 (the second with one slot); TS = 32 with a 1-slot second group in bwd1/bwd3
    "knn_k33": dict(spec=dict(kind=L, cfg=dict(dim=48, edge_dim=2, num_nearest_neighbors=33), B=2, N=150, seed=408,
                              init="xavier", mask="padded"), grads=BOTH),
    # Q = 10 > 8: the shared-memory Q loop pair_bwd2_knn_kernel<T, 16, 0, ...>; k = 2 * 32
    "knn_k64_q10": dict(spec=dict(kind=L, cfg=dict(dim=32, edge_dim=9, num_nearest_neighbors=64), B=2, N=300, seed=409,
                                  init="xavier", mask="random"), grads=BOTH),
    # TS = 1: 128 rows per bwd1 CTA
    "knn_k1": dict(spec=dict(kind=L, cfg=dict(dim=32, num_nearest_neighbors=1), B=2, N=200, seed=410, init="xavier"),
                   grads=BOTH),
    # kNN MP = 32 instantiations
    "knn_mdim32": dict(spec=dict(kind=L, cfg=dict(dim=32, m_dim=32, edge_dim=2, num_nearest_neighbors=17), B=2, N=120, seed=411,
                                 init="xavier"), grads=(F32,)),
    # the two kNN cases of cases.SPECS without a reference-gradient fixture (k = 33; k = 32 with C = 5)
    "spec_knn_k33": dict(spec=cases.SPECS["knn_k33"], grads=BOTH),
    "spec_knn_k32_c5": dict(spec=cases.SPECS["knn_k32_c5"], grads=BOTH),
    # M = 4098 > SN_TABLES_M_MAX: tables through the GEMM; long-K dW; 64 colsum row blocks
    "knn_many_nodes": dict(spec=dict(kind=L, cfg=dict(dim=32, num_nearest_neighbors=8), B=3, N=1366, seed=412, init="xavier"),
                           grads=(F32,)),
    # edge-list backward at k = 40 > 32, with empty slots and one node without neighbours
    "edge_list_k40": dict(spec=dict(kind=L, cfg=dict(dim=24, edge_dim=3, m_pool_method="mean"), B=2, N=90, seed=413,
                                    init="xavier", mask="padded"), grads=BOTH, neighbors=(40, 414)),
    # chained layer gradients at a real size (xavier weights scaled by 0.6: plain xavier overflows exp at depth 3)
    "net_c3_deep": dict(spec=dict(kind=NW, cfg=dict(depth=3, dim=32, num_tokens=21, num_positions=320, num_nearest_neighbors=17),
                                  B=2, N=301, seed=415, init="xavier", mask="padded"), grads=BOTH, weight_scale=0.6),
    # inference only: the tiled dense kernel's shared memory exceeds the budget -> thread-per-pair pair_kernel<T, 16, false>
    "dense_fallback_f32": dict(spec=dict(kind=L, cfg=dict(dim=16, edge_dim=170), B=2, N=40, seed=416, init="xavier",
                                         mask="padded"), grads=(), forward=(F32,)),
    "dense_fallback_f64": dict(spec=dict(kind=L, cfg=dict(dim=16, edge_dim=80), B=2, N=40, seed=417, init="xavier",
                                         mask="padded"), grads=(), forward=(F64,)),
}


@functools.lru_cache(maxsize=None)
def _case(name):
    """-> (case, neighbour lists | None).  Cached: the oracles below are cached per name as well."""
    d = SHAPES[name]
    case = cases.build_case(d["spec"])
    if "weight_scale" in d:
        for k, v in case["params"].items():
            if k.startswith("layers.") and k.endswith(".weight") and np.ndim(v) == 2:
                case["params"][k] = v * d["weight_scale"]
    nb = None
    if "neighbors" in d:
        k, seed = d["neighbors"]
        nb = _edge_list(case["spec"]["B"], case["spec"]["N"], k, seed)
    return case, nb


@functools.lru_cache(maxsize=None)
def _oracle_forward(name):
    case, nb = _case(name)
    if nb is None:
        return cases.run_oracle(case)
    ins = case["inputs"]
    return O.egnn_layer_forward_edge_list(case["params"], case["cfg"], ins["feats"], ins["coors"], nb, ins.get("edges"),
                                          ins.get("mask"))


@functools.lru_cache(maxsize=None)
def _oracle_grads(name):
    case, nb = _case(name)
    if nb is None:
        return cases.flatten_grads(cases.run_oracle_grad(case))
    ins = case["inputs"]
    gf, gx = cases.upstream_grads(case)
    return cases.flatten_grads(G.egnn_layer_backward(case["params"], case["cfg"], ins["feats"], ins["coors"], ins.get("edges"),
                                                     ins.get("mask"), None, gf, gx, neighbors=nb))


def _kw(nb):
    return {} if nb is None else {"neighbors": torch.from_numpy(nb).cuda()}


def _forward(name, dtype):
    case, nb = _case(name)
    mod = util.make_module(case, dtype)
    with torch.no_grad():
        out = util.run_module(mod, case, dtype, **_kw(nb))
    if case["kind"] == L:             # the SIMT kernels, not the bf16 tensor-core path
        assert mod.last_path == ("fp64-simt" if dtype == F64 else "fp32-simt"), mod.last_path
    return out


def _grads(name, dtype):
    case, nb = _case(name)
    return util.module_grads(case, dtype, **_kw(nb))


FWD_PARAMS = [(n, dt) for n, d in SHAPES.items() for dt in d.get("forward", BOTH)]
GRAD_PARAMS = [(n, dt) for n, d in SHAPES.items() for dt in d["grads"]]
_id = lambda dt: "fp64" if dt == F64 else "fp32"


@pytest.mark.gpu
@pytest.mark.parametrize("name,dtype", FWD_PARAMS, ids=[f"{n}-{_id(d)}" for n, d in FWD_PARAMS])
def test_forward_matches_oracle(name, dtype):
    want = _oracle_forward(name)
    got = _forward(name, dtype)
    atol, rtol = (1e-9, 1e-9) if dtype == F64 else (2e-5, 1e-4)
    util.assert_close(got[0], want[0], atol=atol, rtol=rtol, what=f"{name} feats")
    util.assert_close(got[1], want[1], atol=atol, rtol=rtol, what=f"{name} coors")


@pytest.mark.gpu
@pytest.mark.parametrize("saved", [True, False], ids=["saved_pre2", "recompute"])
@pytest.mark.parametrize("name,dtype", GRAD_PARAMS, ids=[f"{n}-{_id(d)}" for n, d in GRAD_PARAMS])
def test_grads_match_oracle(name, dtype, saved, monkeypatch):
    """Saved: bwd1 / bwd2 read the per-pair pre-activations the forward kept (EgnnLayerIO.pre2_out).  Recompute
    (EGNN_B200_SAVE_PAIR_MB=0): dense recomputes them with the register-tiled forward kernel, kNN inside bwd1."""
    if not saved:
        monkeypatch.setenv("EGNN_B200_SAVE_PAIR_MB", "0")
    case, _ = _case(name)
    compare_to = _oracle_grads(name)
    util.compare(_grads(name, dtype), compare_to, util.grad_tol(case, dtype), f"{name} {_id(dtype)} vs oracle")


# ------------------------------------------------------------------ which kernels the matrix runs

def _pat(base, *args):
    """Regex for `base<args...>` in a demangled kernel name; True / False also match 1 / 0."""
    alt = {True: "(?:true|1)", False: "(?:false|0)"}
    parts = [alt[a] if isinstance(a, bool) else re.escape(str(a)) for a in args]
    return re.compile(r"\b" + re.escape(base) + r"<\s*" + r"\s*,\s*".join(parts) + r"\s*>")


REQUIRED = (
    [_pat("pair_bwd1_kernel", t, 16, knn) for t in ("float", "double") for knn in (False, True)]
    + [_pat("pair_bwd1_kernel", "float", 32, knn) for knn in (False, True)]
    + [_pat("pair_bwd2_dense_kernel", t, 16, qr, False) for t in ("float", "double") for qr in (1, 0)]
    + [_pat("pair_bwd2_knn_kernel", t, 16, qr, False) for t in ("float", "double") for qr in (1, 8, 0)]
    + [_pat("pair_bwd2_dense_kernel", "float", 32, 0, False), _pat("pair_bwd2_knn_kernel", "float", 32, 8, False)]
    + [_pat("pair_bwd3_kernel", t, knn) for t in ("float", "double") for knn in (False, True)]
    + [_pat("pair_dense_tiled_kernel", t, 16, 2) for t in ("float", "double")]
    + [_pat("pair_kernel", t, 16, False) for t in ("float", "double")]
    + [_pat("pair_kernel", t, mp, True) for t in ("float", "double") for mp in (16,)] + [_pat("pair_kernel", "float", 32, True)]
    + [_pat(k, t) for k in ("gemm_acc_kernel", "colsum_acc_kernel", "ln_bwd_kernel", "dsilu_mul_kernel",
                            "tables_small_simt_kernel", "node_update_small_simt_kernel", "ln_concat_kernel")
       for t in ("float", "double")]
    + [re.compile(r"\bgemm_nt_kernel<\s*" + t + r"\s*,") for t in ("float", "double")]
)


def _kernels(fn):
    """-> {kernel name: launches} of the CUDA kernels `fn` ran."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.key: e.count for e in prof.key_averages() if e.device_type == torch.autograd.DeviceType.CUDA}


@pytest.mark.gpu
def test_kernel_instantiations_are_exercised():
    def run_matrix():
        for name, d in SHAPES.items():
            for dt in d.get("forward", BOTH):
                _forward(name, dt)
            for dt in d["grads"]:
                _grads(name, dt)

    seen = _kernels(run_matrix)
    missing = [p.pattern for p in REQUIRED if not any(p.search(k) for k in seen)]
    assert not missing, "not launched: " + "; ".join(missing) + "\nlaunched:\n" + "\n".join(sorted(seen))
    # both sides of simt_hsplit: the two-phase dense kernel launches twice per forward, the plain one once
    tiled = lambda name: sum(n for k, n in _kernels(lambda: _forward(name, F64)).items() if "pair_dense_tiled_kernel" in k)
    assert (tiled("c1_hsplit_n64"), tiled("c1_hsplit_n65")) == (2, 1)


# ------------------------------------------------------------------ training preflight

def _nat():
    from egnn_pytorch_b200 import _native, build
    build.build()                     # nvcc cross-compiles sm_100a without a GPU; a no-op when the library is current
    return _native


def _preflight(nat, dtype, knn, m_dim, soft, edge_dim, N=8):
    flags = nat.FLAG_UPDATE_FEATS | nat.FLAG_UPDATE_COORS | (nat.FLAG_SOFT_EDGES if soft else 0)
    d = nat.LayerDesc(abi_version=nat.ABI_VERSION, dtype=nat.DTYPE_F64 if dtype == F64 else nat.DTYPE_F32, B=1, N=N, C=3,
                      dim=8, edge_dim=edge_dim, label_dim=0, num_labels=0, m_dim=m_dim, fourier=0, k=4 if knn else 0,
                      flags=flags, valid_radius=1e30, clamp=0.0, row_begin=0, row_end=0, reserved=0)
    nb = C.c_size_t()
    return nat.load().egnn_layer_backward_workspace_bytes(C.byref(d), C.byref(nb))


def test_backward_preflight_rejects_what_the_backward_cannot_launch():
    """The preflight refuses descriptors whose backward kernels need more dynamic shared memory than the launch
    allows (bwd1 for fp64 with m_dim = 32; the dense bwd2 at edge_dim 48 in fp64), and accepts their neighbours."""
    nat = _nat()
    for knn in (False, True):
        assert _preflight(nat, F64, knn, 32, False, 0) == nat.ERR_UNSUPPORTED, knn
        assert _preflight(nat, F32, knn, 32, False, 0) == 0, knn
        assert _preflight(nat, F64, knn, 16, False, 0) == 0, knn
    assert _preflight(nat, F64, False, 16, False, 47) == 0
    assert _preflight(nat, F64, False, 16, False, 48) == nat.ERR_UNSUPPORTED


SWEEP = [(dt, knn, m, soft) for dt in BOTH for knn in (False, True) for m in (16, 32) for soft in (False, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,knn,m_dim,soft", SWEEP,
                         ids=[f"{_id(dt)}-{'knn' if knn else 'dense'}-m{m}-{'soft' if s else 'hard'}" for dt, knn, m, s in SWEEP])
def test_preflight_accepts_exactly_what_backward_runs(dtype, knn, m_dim, soft):
    """At the last edge_dim the preflight accepts, forward + backward complete and match the gradient oracle; at the
    first one it rejects, the module call raises at the forward (a clean error before any launch)."""
    nat = _nat()
    first_bad = next((e for e in range(0, 257) if _preflight(nat, dtype, knn, m_dim, soft, e) != 0), None)
    assert first_bad is not None and _preflight(nat, dtype, knn, m_dim, soft, first_bad) == nat.ERR_UNSUPPORTED
    for e in sorted({max(0, first_bad - 1), first_bad}):
        cfg = dict(dim=8, m_dim=m_dim, edge_dim=e, soft_edges=soft, num_nearest_neighbors=4 if knn else 0)
        case = cases.build_case(dict(kind=L, cfg=cfg, B=1, N=8, seed=500 + e, init="xavier"))
        if e < first_bad:
            got = util.module_grads(case, dtype)
            want = cases.flatten_grads(cases.run_oracle_grad(case))
            util.compare(got, want, util.grad_tol(case, dtype), f"edge_dim={e}")
        else:
            with pytest.raises(nat.EgnnNativeError, match="egnn_layer_backward_workspace_bytes"):
                util.module_grads(case, dtype)


@pytest.mark.gpu
def test_untrainable_configuration_raises_at_the_forward_call():
    from egnn_pytorch_b200 import EGNN, _native as nat
    mod = EGNN(dim=16, m_dim=32).double().cuda()
    feats = torch.randn(1, 8, 16, dtype=F64, device="cuda", requires_grad=True)
    coors = torch.randn(1, 8, 3, dtype=F64, device="cuda")
    with torch.enable_grad():
        with pytest.raises(nat.EgnnNativeError, match=r"float64.*m_dim=32.*dense"):
            mod(feats, coors)
        with torch.no_grad():
            mod(feats, coors)          # inference with the same module is unaffected
