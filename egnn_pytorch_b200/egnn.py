"""Host-side mirror of the reference's module interface for the EGNN hot path (forward and backward).

`EGNN` and `EGNN_Network` keep the constructor arguments, forward signatures, return values and
state-dict keys of lucidrains/egnn-pytorch (reference egnn_pytorch/egnn_pytorch.py:148-341 and
:343-454), so a reference `state_dict()` loads unchanged -- but `forward` does not execute any
PyTorch arithmetic for the edge step: it packs a POD descriptor and calls the hand-written
sm_100a kernels of libegnn_b200.so through the C ABI (include/egnn_b200.h) on the current CUDA
stream.  PyTorch is used for parameter storage, device memory and streams only.

There is no CPU compute path.  CPU tensors (the reference's own tests pass CPU float64) are
staged to the current CUDA device and the results copied back -- a transport convenience.

Element type -> kernel family
    float64 parameters  -> fp64 SIMT kernels      (parity with the fp64 oracle to ~1e-12)
    float32 parameters  -> fp32 SIMT kernels      ("accurate": the stated-fp32-tolerance path)
    bfloat16 parameters -> tcgen05 bf16 tensor-core kernels with fp32 accumulation ("fast");
                           option combinations the tensor-core kernels do not cover run on the
                           fp32 SIMT kernels instead (still on the GPU; see `last_path`).
`precision='fast'` / `'accurate'` overrides the choice for fp32/bf16 parameters.

Training: when autograd is recording and an input or parameter requires grad, the layer runs as a
`torch.autograd.Function` whose backward is `egnn_layer_backward` -- hand-written recompute-in-backward
kernels (fp32 / fp64; bf16 modules train through the fp32 kernels).  Under `torch.no_grad()` /
`requires_grad_(False)` nothing is saved and the fastest kernels are used.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import os
import warnings

import torch
from torch import nn
import torch.nn.functional as F

from . import _native as nat

__all__ = ["EGNN", "EGNN_Network", "CoorsNorm", "GlobalLinearAttention", "edge_index_to_neighbors"]


def exists(v):
    return v is not None


# ----------------------------------------------------------------------------- runtime helpers

_WORKSPACES: dict = {}
_NULL_CTX = contextlib.nullcontext()


def _workspace(device: torch.device, nbytes: int, stream_handle=None) -> torch.Tensor:
    """Per-(device, stream) scratch arena, grown on demand; the library never allocates."""
    key = (device.index, torch.cuda.current_stream(device).cuda_stream if stream_handle is None else stream_handle)
    ws = _WORKSPACES.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
        _WORKSPACES[key] = ws
    return ws


def _compute_device(t: torch.Tensor) -> torch.device:
    if t.is_cuda:
        return t.device
    if not torch.cuda.is_available():
        raise RuntimeError("egnn_pytorch_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


_KERNEL_DTYPE = {torch.float32: nat.DTYPE_F32, torch.float64: nat.DTYPE_F64, torch.bfloat16: nat.DTYPE_BF16}
_PATH_NAME = {torch.float64: "fp64-simt", torch.float32: "fp32-simt", torch.bfloat16: "bf16-tcgen05"}


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _as_u8(t, dev):
    """bool / uint8 / numeric 0-1 tensor -> contiguous uint8 on `dev`, zero-copy when it already is one."""
    if t is None:
        return None
    if t.device != dev:
        t = t.to(dev, non_blocking=True)
    if t.dtype == torch.bool:
        t = t.view(torch.uint8)
    elif t.dtype != torch.uint8:
        t = t.ne(0).view(torch.uint8)
    return t if t.is_contiguous() else t.contiguous()


def _as(t, dev, dtype):
    """Tensor on `dev` in `dtype`, contiguous; no work when it already is."""
    if t is None:
        return None
    if t.device == dev and t.dtype == dtype and t.is_contiguous():
        return t.detach()
    return t.detach().to(device=dev, dtype=dtype, non_blocking=True).contiguous()


# ----------------------------------------------------------------------------- small modules


class CoorsNorm(nn.Module):
    """Parameter holder for `coors_norm.scale` (reference egnn_pytorch.py:67-77); the
    normalisation x / max(|x|, eps) * scale itself runs inside the fused edge kernel."""

    def __init__(self, eps=1e-8, scale_init=1.0):
        super().__init__()
        self.eps = eps
        self.scale = nn.Parameter(torch.full((1,), float(scale_init)))


def _mlp(d_in, d_hidden, d_out, dropout, final_act=False):
    """Linear -> (Dropout|Identity) -> SiLU -> Linear [-> SiLU]; the Sequential indices (0 and 3)
    are part of the state-dict contract (reference :178-184, :196-201, :203-208)."""
    mods = [nn.Linear(d_in, d_hidden), nn.Dropout(dropout) if dropout > 0 else nn.Identity(), nn.SiLU(),
            nn.Linear(d_hidden, d_out)]
    if final_act:
        mods.append(nn.SiLU())
    return nn.Sequential(*mods)


# ----------------------------------------------------------------------------- autograd bridge


class _EGNNLayerFunction(torch.autograd.Function):
    """forward = egnn_layer_forward on a private workspace that is kept for backward;
    backward = egnn_layer_backward (what autograd derives from reference egnn_pytorch.py:224-341)."""

    @staticmethod
    def forward(ctx, run, feats, coors, edges, label_emb, *params):
        f_out, x_out, saved = run()
        ctx.saved = saved
        tensors = (feats, coors, edges, label_emb) + params
        ctx.meta = [(t.dtype, t.device) if t is not None else None for t in tensors]
        # the saved state aliases the inputs and (same device / dtype) the live parameters: remember their versions so
        # that an in-place edit between forward and backward is reported instead of silently differentiated
        ctx.versions = [(t, t._version) for t in tensors if t is not None]
        return f_out, x_out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_f, g_x):
        sv = ctx.saved
        if sv is None:
            raise RuntimeError("egnn_pytorch_b200: backward through this EGNN layer a second time: the saved forward workspace "
                               "is released after the first backward (retain_graph=True is not supported; run the forward again)")
        for t, v in ctx.versions:
            if t._version != v:
                raise RuntimeError("egnn_pytorch_b200: a tensor needed for the gradient of an EGNN layer (an input or a parameter) "
                                   "was modified in place between forward and backward")
        lib, dev, kdt, cdt = nat.load(), sv["dev"], sv["kdt"], sv["cdt"]
        T = sv["tensors"]
        with torch.cuda.device(dev):
            stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            g_f, g_x = _as(g_f, dev, kdt), _as(g_x, dev, cdt)
            gw = {f: torch.empty_like(T[f]) for f in nat.WEIGHT_FIELDS if f in T}
            g_feats, g_coors = torch.empty_like(sv["f_in"]), torch.empty_like(sv["x_in"])
            g_edges = torch.empty_like(sv["e_in"]) if (sv["e_in"] is not None and ctx.needs_input_grad[3]) else None
            grads = nat.LayerGrads(g_feats_out=g_f.data_ptr(), g_coors_out=g_x.data_ptr(), g_feats=g_feats.data_ptr(),
                                   g_coors=g_coors.data_ptr(), g_edges=None if g_edges is None else g_edges.data_ptr(),
                                   w=nat.LayerWeightGrads(**{f: t.data_ptr() for f, t in gw.items()}))
            nb = C.c_size_t()
            nat.check("egnn_layer_backward_workspace_bytes",
                      lib.egnn_layer_backward_workspace_bytes(C.byref(sv["desc"]), C.byref(nb)))
            ws = _workspace(dev, nb.value)
            nat.check("egnn_layer_backward",
                      lib.egnn_layer_backward(C.byref(sv["desc"]), C.byref(sv["w"]), _ptr(sv["packed"]), C.byref(sv["io"]),
                                              _ptr(sv["ws"]), C.byref(grads), _ptr(ws), ws.numel(), stream))
        ctx.saved = None
        back = lambda g, m: None if (g is None or m is None) else g.to(device=m[1], dtype=m[0])
        out = [None, back(g_feats, ctx.meta[0]), back(g_coors, ctx.meta[1]), back(g_edges, ctx.meta[2]),
               back(gw.get("label_emb"), ctx.meta[3])]
        for f, m in zip(sv["param_fields"], ctx.meta[4:]):
            out.append(back(gw.get(f), m))
        return tuple(g if need else None for g, need in zip(out, ctx.needs_input_grad))


# ----------------------------------------------------------------------------- the layer


class EGNN(nn.Module):
    """Drop-in for `egnn_pytorch.EGNN` (reference egnn_pytorch.py:148-341)."""

    def __init__(self, dim, edge_dim=0, m_dim=16, fourier_features=0, num_nearest_neighbors=0, dropout=0.0,
                 init_eps=1e-3, norm_feats=False, norm_coors=False, norm_coors_scale_init=1e-2,
                 update_feats=True, update_coors=True, only_sparse_neighbors=False, valid_radius=float("inf"),
                 m_pool_method="sum", soft_edges=False, coor_weights_clamp_value=None, precision="auto"):
        super().__init__()
        assert m_pool_method in {"sum", "mean"}, "pool method must be either sum or mean"
        assert update_feats or update_coors, "you must update either features, coordinates, or both"
        assert precision in {"auto", "accurate", "fast"}
        self.dim, self.edge_dim, self.m_dim = dim, edge_dim, m_dim
        self.fourier_features = fourier_features
        edge_input_dim = fourier_features * 2 + dim * 2 + edge_dim + 1
        self.edge_mlp = _mlp(edge_input_dim, edge_input_dim * 2, m_dim, dropout, final_act=True)
        self.edge_gate = nn.Sequential(nn.Linear(m_dim, 1), nn.Sigmoid()) if soft_edges else None
        self.node_norm = nn.LayerNorm(dim) if norm_feats else nn.Identity()
        self.coors_norm = CoorsNorm(scale_init=norm_coors_scale_init) if norm_coors else nn.Identity()
        self.m_pool_method = m_pool_method
        self.node_mlp = _mlp(dim + m_dim, dim * 2, dim, dropout) if update_feats else None
        self.coors_mlp = _mlp(m_dim, m_dim * 4, 1, dropout) if update_coors else None
        self.num_nearest_neighbors = num_nearest_neighbors
        self.only_sparse_neighbors = only_sparse_neighbors
        self.valid_radius = valid_radius
        self.coor_weights_clamp_value = coor_weights_clamp_value
        self.dropout_p = dropout
        self.init_eps = init_eps
        self.precision = precision
        self.last_path = None          # 'fp64-simt' | 'fp32-simt' | 'bf16-tcgen05' of the last call
        self.cache_policy = "version"  # 'version' | 'always' -- see invalidate_cache()
        self._stage = {}
        self._tc_unsupported = set()
        self._call_cache = {}
        self.apply(self._init)

    def _init(self, module):
        if type(module) is nn.Linear:
            nn.init.normal_(module.weight, std=self.init_eps)      # reference :219-222

    # -------------------------------------------------------------- parameter staging
    def _state_fields(self):
        """[(EgnnLayerWeights field, Parameter)], cached; rebuilt if a Parameter object is replaced."""
        cache = self.__dict__.get("_fields_cache")
        if cache is not None and all(mod._parameters.get(name) is p for mod, name, _, p in cache):
            return cache
        cache = []
        for mname, mod in self.named_modules():
            for pname, p in mod._parameters.items():
                key = f"{mname}.{pname}" if mname else pname
                f = nat.STATE_KEY_TO_FIELD.get(key)
                if f is not None and p is not None:
                    cache.append((mod, pname, f, p))
        self.__dict__["_fields_cache"] = cache
        return cache

    def invalidate_cache(self):
        """Drop every staged / packed copy of the parameters (they are rebuilt on the next call).

        The caches are keyed on (storage pointer, tensor version) of each parameter.  Writes that go THROUGH
        `.data` (`p.data.copy_(master)`, the master->model copy of apex / DeepSpeed / Megatron-style mixed
        precision, some EMA loops) do not bump the version counter, so after such a write call this method -- or
        set `cache_policy = "always"` to re-stage and re-pack on every forward (one small kernel per layer).
        In training mode (`module.training` with a parameter that requires grad) the layer always re-packs."""
        self._stage = {}
        self._call_cache = {}
        self.__dict__.pop("_fields_cache", None)

    def _staged(self, device, dtype):
        fields = self._state_fields()
        sig = [x for _, _, _, p in fields for x in (p.data_ptr(), p._version)]
        key = (device, dtype)
        st = self._stage.get(key)
        always = self.cache_policy == "always" or (self.training and any(p.requires_grad for _, _, _, p in fields))
        if st is None or st["sig"] != sig or always:
            with torch.no_grad():
                tensors = {f: p.detach().to(device=device, dtype=dtype).contiguous() for _, _, f, p in fields}
            st = dict(sig=sig, tensors=tensors, packed={}, wstruct={})
            self._stage[key] = st
        return st

    def _flags(self):
        fl = self.__dict__.get("_flags_cache")
        if fl is None:                           # which sub-modules exist is fixed by the constructor
            fl = 0
            if isinstance(self.node_norm, nn.LayerNorm): fl |= nat.FLAG_NORM_FEATS
            if isinstance(self.coors_norm, CoorsNorm): fl |= nat.FLAG_NORM_COORS
            if self.node_mlp is not None: fl |= nat.FLAG_UPDATE_FEATS
            if self.coors_mlp is not None: fl |= nat.FLAG_UPDATE_COORS
            if self.edge_gate is not None: fl |= nat.FLAG_SOFT_EDGES
            self.__dict__["_flags_cache"] = fl
        # plain attributes a user may change between calls are read every time
        if self.m_pool_method == "mean": fl |= nat.FLAG_POOL_MEAN
        if self.coor_weights_clamp_value is not None: fl |= nat.FLAG_CLAMP
        return fl

    def _kernel_dtype(self):
        pd = self._modules["edge_mlp"]._modules["0"]._parameters["weight"].dtype     # edge_mlp[0].weight without three __getattr__ hops
        if pd == torch.float64:
            return torch.float64
        prec = os.environ.get("EGNN_B200_PRECISION", self.precision)
        if prec == "fast" or (prec == "auto" and pd == torch.bfloat16):
            return torch.bfloat16
        return torch.float32

    # -------------------------------------------------------------- forward
    def forward(self, feats, coors, edges=None, mask=None, adj_mat=None, *, neighbors=None, _edge_labels=None,
                _label_emb=None, _k_hint=None, _rows=None):
        """Reference signature `forward(feats, coors, edges=None, mask=None, adj_mat=None)` (egnn_pytorch.py:224).

        `neighbors` (additive, keyword-only): int tensor [B, N, k] of neighbour indices, -1 = empty slot.  When
        given, the layer runs on exactly these edges and the O(N^2) distance / top-k pass is skipped -- the
        edge-list mode of SURVEY.md section 8(f) (`edge_index_to_neighbors` converts a PyG-style edge_index)."""
        if torch.is_grad_enabled():             # (the parameter scan is skipped entirely under torch.no_grad())
            fields = self._state_fields()
            if (feats.requires_grad or coors.requires_grad or (edges is not None and edges.requires_grad) or
                    (_label_emb is not None and _label_emb.requires_grad) or any(p.requires_grad for _, _, _, p in fields)):
                return self._forward_train(fields, feats, coors, edges, mask, adj_mat, neighbors, _edge_labels, _label_emb,
                                           _k_hint, _rows)
            with torch.no_grad():
                return self._forward_impl(feats, coors, edges, mask, adj_mat, neighbors, _edge_labels, _label_emb, _k_hint,
                                          _rows)
        return self._forward_impl(feats, coors, edges, mask, adj_mat, neighbors, _edge_labels, _label_emb, _k_hint, _rows)

    def _forward_train(self, fields, feats, coors, edges, mask, adj_mat, neighbors, labels, label_emb, k_hint, rows):
        if rows is not None:
            raise NotImplementedError("a row range (_rows) cannot be differentiated: call it under torch.no_grad() for "
                                      "inference, or shard the batch (parallel.batch_sharded_call) for training")
        params = [p for _, _, _, p in fields]

        def run():
            return self._forward_impl(feats, coors, edges, mask, adj_mat, neighbors, labels, label_emb, k_hint, None,
                                      train=True, param_fields=[f for _, _, f, _ in fields])

        return _EGNNLayerFunction.apply(run, feats, coors, edges, label_emb, *params)

    def _forward_impl(self, feats, coors, edges, mask, adj_mat, neighbors, _edge_labels, _label_emb, _k_hint, _rows,
                      train=False, param_fields=None):
        lib = nat.load()
        dev = _compute_device(feats)
        b, n, d = feats.shape
        assert d == self.dim, f"feature width {d} != dim {self.dim}"
        c = coors.shape[-1]
        kdt = self._kernel_dtype()
        # nn.Dropout of the three MLPs (reference :176-208) is active in training mode only, grad or no grad -- like
        # the reference.  The kernels regenerate the masks from (seed, element index) in forward and backward; the seed
        # is drawn per call from torch's CPU generator, so torch.manual_seed makes a run reproducible.
        drop_p = float(self.dropout_p) if (self.training and self.dropout_p > 0) else 0.0
        if (train or drop_p > 0) and kdt == torch.bfloat16:
            kdt = torch.float32                 # the tensor-core kernels are forward-only and have no dropout
        label_dim = 0 if _label_emb is None else _label_emb.shape[1]
        cont_edge_dim = self.edge_dim - label_dim
        assert (edges is None) == (cont_edge_dim == 0), "edges must be given iff edge_dim > 0"

        use_nearest = self.num_nearest_neighbors > 0 or self.only_sparse_neighbors          # reference :230
        adj_u8 = None
        k = 0
        flags = self._flags()
        nbr = None
        if neighbors is not None:
            assert neighbors.dim() == 3 and neighbors.shape[:2] == (b, n), "neighbors must be [B, N, k]"
            nbr = neighbors.to(device=dev, dtype=torch.int32).contiguous()
            k = nbr.shape[-1]
            if not (0 < k <= n):
                raise RuntimeError(f"neighbour lists need 0 < k <= N, got k={k}, N={n}")
        elif use_nearest:
            k = self.num_nearest_neighbors
            if exists(adj_mat):
                adj_u8 = _as_u8(adj_mat, dev)
                if adj_u8.dim() == 3:
                    flags |= nat.FLAG_ADJ_BATCHED
                if self.only_sparse_neighbors:
                    flags |= nat.FLAG_ONLY_SPARSE                                    # valid_radius := 0 (:250)
                    # reference :249 -- one host sync, diagonal still counted
                    k = int(_k_hint) if _k_hint is not None else int(adj_u8.sum(dim=-1, dtype=torch.int32).max().item())
            if not (0 < k <= n):
                raise RuntimeError(f"number of neighbours k={k} must satisfy 0 < k <= N={n} (torch.topk would raise)")

        cfg_key = (c, k > 0, min(k, 33), cont_edge_dim, label_dim, _rows is None)
        if kdt == torch.bfloat16 and cfg_key in self._tc_unsupported:
            kdt = torch.float32
        try:
            return self._run(lib, dev, kdt, feats, coors, edges, mask, adj_u8, _edge_labels, _label_emb,
                             b, n, c, k, flags, cont_edge_dim, label_dim, _rows, nbr, train, param_fields, drop_p)
        except nat.EgnnNativeError as e:
            if e.code != nat.ERR_UNSUPPORTED or kdt != torch.bfloat16:
                raise
        # the tensor-core kernels do not cover this option set: fp32 SIMT kernels (still on the GPU); remembered
        self._tc_unsupported.add(cfg_key)
        warnings.warn(f"egnn_pytorch_b200: the bf16 tensor-core kernels do not cover this configuration (C={c}, k={k}, "
                      f"edge_dim={cont_edge_dim}, label_dim={label_dim}, m_dim={self.m_dim}, fourier={self.fourier_features}); "
                      f"running the fp32 SIMT kernels instead (about 5x slower, same results to fp32 accuracy)", UserWarning,
                      stacklevel=3)
        return self._run(lib, dev, torch.float32, feats, coors, edges, mask, adj_u8, _edge_labels, _label_emb,
                         b, n, c, k, flags, cont_edge_dim, label_dim, _rows, nbr)

    def _run(self, lib, dev, kdt, feats, coors, edges, mask, adj_u8, labels, label_emb, b, n, c, k, flags,
             cont_edge_dim, label_dim, rows, nbr=None, train=False, param_fields=None, drop_p=0.0):
        cdt = torch.float64 if kdt == torch.float64 else torch.float32
        st = self._staged(dev, kdt)
        T = dict(st["tensors"])
        lab_w = None
        if label_emb is not None:
            lab_w = st.get("lab_keepalive")
            if lab_w is None or st.get("lab_sig") != (label_emb.data_ptr(), label_emb._version):
                lab_w = label_emb.detach().to(device=dev, dtype=kdt).contiguous()
                st["lab_sig"] = (label_emb.data_ptr(), label_emb._version)
                st["wstruct"] = {}
                st["packed"] = {}
            T["label_emb"] = lab_w

        ckey = (kdt, b, n, c, k, flags, cont_edge_dim, label_dim, 0 if label_emb is None else label_emb.shape[0], rows,
                float(self.valid_radius), float(self.coor_weights_clamp_value or 0.0))
        cc = self._call_cache.get(ckey)
        if cc is None:
            desc = nat.LayerDesc(
                abi_version=nat.ABI_VERSION, dtype=_KERNEL_DTYPE[kdt], B=b, N=n, C=c, dim=self.dim,
                edge_dim=cont_edge_dim, label_dim=label_dim, num_labels=0 if label_emb is None else label_emb.shape[0],
                m_dim=self.m_dim, fourier=self.fourier_features, k=k, flags=flags,
                valid_radius=float(self.valid_radius), clamp=float(self.coor_weights_clamp_value or 0.0),
                row_begin=0 if rows is None else rows[0], row_end=0 if rows is None else rows[1], reserved=0,
                dropout_p=0.0, dropout_seed=0)
            nb = C.c_size_t()
            nat.check("egnn_layer_workspace_bytes", lib.egnn_layer_workspace_bytes(C.byref(desc), C.byref(nb)))
            cc = (desc, nb.value)
            if len(self._call_cache) > 64:
                self._call_cache.clear()
            self._call_cache[ckey] = cc
        desc, ws_bytes = cc
        if drop_p > 0:                               # per-call copy: fresh seed, kept with the saved state for backward
            d2 = nat.LayerDesc()
            C.memmove(C.byref(d2), C.byref(desc), C.sizeof(nat.LayerDesc))
            d2.dropout_p = drop_p
            d2.dropout_seed = int(torch.randint(0, 2 ** 62, (1,)).item())
            desc = d2
        wkey = None if lab_w is None else (label_emb.data_ptr(), label_emb._version)
        w = st["wstruct"].get(wkey)
        if w is None:
            w = nat.LayerWeights(**{f: (T[f].data_ptr() if f in T else None) for f in nat.WEIGHT_FIELDS})
            st["wstruct"] = {wkey: w}
            st["lab_keepalive"] = lab_w

        stream_handle = torch.cuda.current_stream(dev).cuda_stream
        stream = C.c_void_p(stream_handle)
        ctx = _NULL_CTX if torch.cuda.current_device() == dev.index else torch.cuda.device(dev)
        with ctx:
            # packed parameters, cached until a parameter changes
            pkey = (label_dim, 0 if lab_w is None else (label_emb.data_ptr(), label_emb._version))
            packed = st["packed"].get(pkey)
            if packed is None:
                nb = C.c_size_t()
                nat.check("egnn_layer_packed_bytes", lib.egnn_layer_packed_bytes(C.byref(desc), C.byref(nb)))
                packed = torch.empty(nb.value, dtype=torch.uint8, device=dev)
                nat.check("egnn_layer_pack_weights",
                          lib.egnn_layer_pack_weights(C.byref(desc), C.byref(w), _ptr(packed), nb.value, stream))
                st["packed"] = {pkey: packed}

            f_in, x_in, e_in = _as(feats, dev, kdt), _as(coors, dev, cdt), _as(edges, dev, kdt)
            m_in, l_in = _as_u8(mask, dev), _as_u8(labels, dev)
            f_out = torch.empty_like(f_in)
            x_out = torch.empty_like(x_in)
            if rows is not None:       # rows outside the range keep the input values
                f_out.copy_(f_in)
                x_out.copy_(x_in)
            # training: keep the per-pair pre-activations of edge_mlp's second SiLU (64 B per pair in fp32) so
            # that backward need not recompute them, unless that exceeds EGNN_B200_SAVE_PAIR_MB (default 1024)
            pre2 = None
            if train:
                mp = 16 if self.m_dim <= 16 else 32
                nbytes = b * n * (k if k > 0 else n) * mp * f_in.element_size()
                if nbytes <= float(os.environ.get("EGNN_B200_SAVE_PAIR_MB", "1024")) * 2 ** 20:
                    pre2 = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            # the library reads EgnnLayerIO during the call only: inference re-fills one struct per layer, training
            # (which keeps it with the saved state) gets its own
            io = nat.LayerIO() if train else self.__dict__.get("_io_scratch")
            if io is None:
                io = self.__dict__["_io_scratch"] = nat.LayerIO()
            io.feats = f_in.data_ptr(); io.coors = x_in.data_ptr()
            io.edges = None if e_in is None else e_in.data_ptr()
            io.edge_labels = None if l_in is None else l_in.data_ptr()
            io.mask = None if m_in is None else m_in.data_ptr()
            io.adj = None if adj_u8 is None else adj_u8.data_ptr()
            io.feats_out = f_out.data_ptr(); io.coors_out = x_out.data_ptr()
            io.nbr_idx = None if nbr is None else nbr.data_ptr()
            io.pre2_out = None if pre2 is None else pre2.data_ptr()
            if train:     # preflight: configurations the backward kernels cannot run fail HERE, before the forward launches
                nbb = C.c_size_t()
                rc = lib.egnn_layer_backward_workspace_bytes(C.byref(desc), C.byref(nbb))
                if rc == nat.ERR_UNSUPPORTED:
                    raise nat.EgnnNativeError(
                        "egnn_layer_backward_workspace_bytes", rc,
                        f"the backward kernels cannot train this layer ({str(kdt).replace('torch.', '')}, dim={self.dim}, "
                        f"m_dim={self.m_dim}, edge_dim={self.edge_dim}, fourier_features={self.fourier_features}, "
                        f"{f'k={k} neighbours' if k > 0 else 'dense'}, soft_edges={self.edge_gate is not None}"
                        f"{'' if rows is None else f', rows {rows[0]}:{rows[1]}'}); see DESIGN.md section 9 'Limits'")
                nat.check("egnn_layer_backward_workspace_bytes", rc)
            # training keeps the workspace (per-node tables, pooled messages, neighbour lists) for backward
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev) if train else _workspace(dev, ws_bytes, stream_handle)
            nat.check("egnn_layer_forward",
                      lib.egnn_layer_forward(C.byref(desc), C.byref(w), _ptr(packed), C.byref(io), _ptr(ws),
                                             ws.numel(), stream))
        object.__setattr__(self, "last_path", _PATH_NAME[kdt])
        outs = (f_out if (f_out.dtype == feats.dtype and f_out.device == feats.device) else f_out.to(device=feats.device, dtype=feats.dtype),
                x_out if (x_out.dtype == coors.dtype and x_out.device == coors.device) else x_out.to(device=coors.device, dtype=coors.dtype))
        if not train:
            return outs
        saved = dict(dev=dev, kdt=kdt, cdt=cdt, desc=desc, w=w, packed=packed, io=io, ws=ws, tensors=T,
                     f_in=f_in, x_in=x_in, e_in=e_in, param_fields=param_fields,
                     keep=(m_in, l_in, adj_u8, nbr, lab_w, pre2))      # everything io points at stays alive
        return outs + (saved,)


def edge_index_to_neighbors(edge_index, num_nodes, k=None):
    """PyG-style `edge_index` [2, E] (messages flow source j = edge_index[0] -> target i = edge_index[1], one graph)
    -> padded neighbour lists [1, N, k] for `EGNN.forward(..., neighbors=...)`; -1 marks empty slots.  Glue code:
    a stable sort by target node, nothing on the hot path."""
    src, dst = edge_index[0].long(), edge_index[1].long()
    order = torch.argsort(dst, stable=True)
    src, dst = src[order], dst[order]
    deg = torch.bincount(dst, minlength=num_nodes)
    kmax = int(deg.max().item()) if k is None else k
    start = torch.cumsum(deg, 0) - deg
    slot = torch.arange(src.numel(), device=src.device) - start[dst]
    out = torch.full((num_nodes, kmax), -1, dtype=torch.int32, device=src.device)
    keep = slot < kmax
    out[dst[keep], slot[keep]] = src[keep].to(torch.int32)
    return out.unsqueeze(0)


# ----------------------------------------------------------------------------- global attention


class _Attention(nn.Module):
    """Parameter holder (+ autograd path) of the multi-head softmax attention inside GlobalLinearAttention
    (reference egnn_pytorch.py:81-110): `to_q`, `to_kv` without bias, `to_out` with bias."""

    def __init__(self, dim, heads=8, dim_head=64):
        super().__init__()
        inner = heads * dim_head
        self.heads, self.dim_head = heads, dim_head
        self.to_q = nn.Linear(dim, inner, bias=False)
        self.to_kv = nn.Linear(dim, inner * 2, bias=False)
        self.to_out = nn.Linear(inner, dim)

    def forward(self, x, context, mask=None):
        """Training path (PyTorch autograd).  Masked keys get the most negative finite score BEFORE the softmax, like the
        reference (:101-104), so a fully masked graph attends uniformly instead of producing NaN."""
        h = self.heads
        q = self.to_q(x)
        k, v = self.to_kv(context).chunk(2, dim=-1)
        split = lambda t: t.unflatten(-1, (h, -1)).transpose(1, 2)
        q, k, v = split(q), split(k), split(v)
        dots = (q @ k.transpose(-1, -2)) * self.dim_head ** -0.5
        if mask is not None:
            dots = dots.masked_fill(~mask[:, None, None, :].to(torch.bool), -torch.finfo(dots.dtype).max)
        out = dots.softmax(dim=-1) @ v
        return self.to_out(out.transpose(1, 2).flatten(-2))


class GlobalLinearAttention(nn.Module):
    """Induced-set attention between the nodes and a few global tokens (reference egnn_pytorch.py:112-144).

    Inference (no autograd recording): ONE call of `egnn_global_attn_forward` (csrc/global_attn.cu) on staged fp32 / fp64
    copies of the parameters -- the module itself is never moved.  When a gradient is required the same arithmetic runs
    through PyTorch autograd (the hand-written backward of SURVEY.md section 8(f) covers the EGNN layers only)."""

    def __init__(self, *, dim, heads=8, dim_head=64):
        super().__init__()
        self.dim, self.heads, self.dim_head = dim, heads, dim_head
        self.norm_seq = nn.LayerNorm(dim)
        self.norm_queries = nn.LayerNorm(dim)
        self.attn1 = _Attention(dim, heads, dim_head)
        self.attn2 = _Attention(dim, heads, dim_head)
        self.ff = nn.Sequential(nn.LayerNorm(dim), nn.Linear(dim, dim * 4), nn.GELU(), nn.Linear(dim * 4, dim))
        self._stage = {}

    def _forward_autograd(self, x, queries, mask=None):
        nx, nq = self.norm_seq(x), self.norm_queries(queries)
        induced = self.attn1(nq, nx, mask=mask)
        x = self.attn2(nx, induced) + x
        queries = induced + queries
        return self.ff(x) + x, queries

    def _staged(self, device, dtype):
        named = [(k, p) for k, p in self.named_parameters() if k in nat.GA_STATE_KEY_TO_FIELD]
        sig = tuple((p.data_ptr(), p._version) for _, p in named)
        st = self._stage.get((device, dtype))
        if st is None or st[0] != sig:
            with torch.no_grad():
                tensors = {nat.GA_STATE_KEY_TO_FIELD[k]: p.detach().to(device=device, dtype=dtype).contiguous() for k, p in named}
            w = nat.GlobalAttnWeights(**{f: t.data_ptr() for f, t in tensors.items()})
            st = (sig, tensors, w)
            self._stage[(device, dtype)] = st
        return st

    def invalidate_cache(self):
        self._stage = {}

    def forward(self, x, queries, mask=None):
        needs_grad = torch.is_grad_enabled() and (x.requires_grad or queries.requires_grad or
                                                  any(p.requires_grad for p in self.parameters()))
        if needs_grad:
            dev = x.device
            if any(p.device != dev for p in self.parameters()):
                raise RuntimeError("training GlobalLinearAttention needs the module on the device of its inputs")
            return self._forward_autograd(x, queries, mask)
        lib = nat.load()
        dev = _compute_device(x)
        kdt = torch.float64 if x.dtype == torch.float64 else torch.float32
        _, _, w = self._staged(dev, kdt)
        b, n, d = x.shape
        t = queries.shape[1]
        x_in, q_in, m_in = _as(x, dev, kdt), _as(queries, dev, kdt), _as_u8(mask, dev)
        x_out, q_out = torch.empty_like(x_in), torch.empty_like(q_in)
        desc = nat.GlobalAttnDesc(abi_version=nat.ABI_VERSION, dtype=_KERNEL_DTYPE[kdt], B=b, N=n, T=t, dim=d, heads=self.heads,
                                  dim_head=self.dim_head)
        nb = C.c_size_t()
        nat.check("egnn_global_attn_workspace_bytes", lib.egnn_global_attn_workspace_bytes(C.byref(desc), C.byref(nb)))
        io = nat.GlobalAttnIO(x=x_in.data_ptr(), queries=q_in.data_ptr(), mask=None if m_in is None else m_in.data_ptr(),
                              x_out=x_out.data_ptr(), queries_out=q_out.data_ptr())
        with torch.cuda.device(dev):
            ws = _workspace(dev, nb.value)
            nat.check("egnn_global_attn_forward",
                      lib.egnn_global_attn_forward(C.byref(desc), C.byref(w), C.byref(io), _ptr(ws), ws.numel(),
                                                   C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
        return x_out.to(device=x.device, dtype=x.dtype), q_out.to(device=queries.device, dtype=queries.dtype)


# ----------------------------------------------------------------------------- the network


class EGNN_Network(nn.Module):
    """Drop-in for `egnn_pytorch.EGNN_Network` (reference egnn_pytorch.py:343-454).

    Differences in mechanism, not in results: the N-th degree adjacency is expanded on bit-packed
    rows by `egnn_adj_expand` instead of dense `A @ A` (:425), and the adjacency-degree embedding
    is never materialised as a [B,N,N,adj_dim] tensor (:430-432) -- layers receive the uint8 degree
    labels and fold `adj_emb.weight` into a [num_degrees+1, H] table."""

    def __init__(self, *, depth, dim, num_tokens=None, num_edge_tokens=None, num_positions=None, edge_dim=0,
                 num_adj_degrees=None, adj_dim=0, global_linear_attn_every=0, global_linear_attn_heads=8,
                 global_linear_attn_dim_head=64, num_global_tokens=4, **kwargs):
        super().__init__()
        assert not (exists(num_adj_degrees) and num_adj_degrees < 1), "make sure adjacent degrees is greater than 1"
        self.num_positions = num_positions
        self.token_emb = nn.Embedding(num_tokens, dim) if exists(num_tokens) else None
        self.pos_emb = nn.Embedding(num_positions, dim) if exists(num_positions) else None
        self.edge_emb = nn.Embedding(num_edge_tokens, edge_dim) if exists(num_edge_tokens) else None
        self.has_edges = edge_dim > 0
        self.num_adj_degrees = num_adj_degrees
        self.adj_emb = nn.Embedding(num_adj_degrees + 1, adj_dim) if exists(num_adj_degrees) and adj_dim > 0 else None
        edge_dim = edge_dim if self.has_edges else 0
        adj_dim = adj_dim if exists(num_adj_degrees) else 0
        has_global_attn = global_linear_attn_every > 0
        self.global_tokens = nn.Parameter(torch.randn(num_global_tokens, dim)) if has_global_attn else None
        self.layers = nn.ModuleList()
        for ind in range(depth):
            is_global = has_global_attn and (ind % global_linear_attn_every) == 0
            self.layers.append(nn.ModuleList([
                GlobalLinearAttention(dim=dim, heads=global_linear_attn_heads,
                                      dim_head=global_linear_attn_dim_head) if is_global else None,
                EGNN(dim=dim, edge_dim=edge_dim + adj_dim, norm_feats=True, **kwargs),
            ]))

    def forward(self, feats, coors, adj_mat=None, edges=None, mask=None, return_coor_changes=False):
        lib = nat.load()
        out_dev = coors.device
        dev = _compute_device(coors)
        b = feats.shape[0]
        feats, coors = feats.to(dev), coors.to(dev)
        adj_mat = None if adj_mat is None else adj_mat.to(dev)
        edges = None if edges is None else edges.to(dev)
        mask = None if mask is None else mask.to(dev)

        def staged(emb):
            return emb.weight if emb.weight.device == dev else emb.weight.to(dev)

        if exists(self.pos_emb):
            n = feats.shape[1]
            assert n <= self.num_positions, \
                f"given sequence length {n} must be less than the number of positions {self.num_positions} set at init"
        emb_grad = torch.is_grad_enabled() and any(e is not None and e.weight.requires_grad for e in (self.token_emb, self.pos_emb))
        if exists(self.token_emb) and not emb_grad and self.token_emb.weight.dtype in _KERNEL_DTYPE:
            # token + positional embedding in ONE launch (egnn_embed_nodes) instead of embedding, arange, embedding, add
            tw = staged(self.token_emb)
            pw = staged(self.pos_emb) if exists(self.pos_emb) else None
            tok = feats.to(torch.int64).contiguous()
            n = tok.shape[1]
            feats = torch.empty((b, n, tw.shape[1]), dtype=tw.dtype, device=dev)
            with (_NULL_CTX if torch.cuda.current_device() == dev.index else torch.cuda.device(dev)):
                nat.check("egnn_embed_nodes", lib.egnn_embed_nodes(
                    _KERNEL_DTYPE[tw.dtype], b, n, tw.shape[1], tw.shape[0], _ptr(tok), _ptr(tw), _ptr(pw), _ptr(feats),
                    C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
        else:                                        # training through the embedding tables: PyTorch autograd
            if exists(self.token_emb):
                feats = F.embedding(feats, staged(self.token_emb))                   # reference :401-402
            if exists(self.pos_emb):
                feats = feats + staged(self.pos_emb)[:feats.shape[1]].unsqueeze(0)   # :404-408
        if exists(edges) and exists(self.edge_emb):
            edges = F.embedding(edges, staged(self.edge_emb))                        # :410-411

        labels = label_emb = k_hint = nbr_lists = None
        if exists(self.num_adj_degrees):
            assert exists(adj_mat), "adjacency matrix must be passed in (keyword argument adj_mat)"
            # the expansion depends on the adjacency only: cached per (storage, version), which also keeps the
            # reference's host sync (:249) out of repeated calls and makes the forward CUDA-graph capturable
            akey = (adj_mat.data_ptr(), adj_mat._version, tuple(adj_mat.shape), b, self.num_adj_degrees)
            cached = self.__dict__.get("_adj_cache")
            if cached is None or cached[0] != akey:
                n = adj_mat.shape[-1]
                adj_in = adj_mat.ne(0).to(torch.uint8).contiguous()
                adj_out = torch.empty((b, n, n), dtype=torch.uint8, device=dev)
                lab = torch.empty((b, n, n), dtype=torch.uint8, device=dev)
                max_sum = torch.zeros(1, dtype=torch.int32, device=dev)
                nb = C.c_size_t()
                nat.check("egnn_adj_workspace_bytes", lib.egnn_adj_workspace_bytes(b, n, C.byref(nb)))
                with torch.cuda.device(dev):
                    ws = _workspace(dev, nb.value)
                    nat.check("egnn_adj_expand", lib.egnn_adj_expand(
                        b, n, self.num_adj_degrees, _ptr(adj_in), 1 if adj_in.dim() == 3 else 0, _ptr(adj_out), _ptr(lab),
                        _ptr(max_sum), _ptr(ws), ws.numel(), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
                kmax = int(max_sum.item()) if self.layers[0][1].only_sparse_neighbors else None   # the reference's sync at :249
                # only_sparse_neighbors with a node mask: the surviving slots of every layer's top-k are the node and its
                # adjacent nodes (valid_radius = 0, :250, :296) -- lists that depend on the adjacency only.  Built once
                # here (egnn_adj_neighbors) and handed to every layer instead of one adjacency scan per layer.
                lists = None
                if kmax is not None and 0 < kmax <= n and os.environ.get("EGNN_B200_NO_LIST_CACHE") != "1":
                    lists = torch.empty((b, n, kmax), dtype=torch.int32, device=dev)
                    with torch.cuda.device(dev):
                        nat.check("egnn_adj_neighbors", lib.egnn_adj_neighbors(
                            b, n, kmax, _ptr(adj_out), 1, _ptr(lists), None, C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
                cached = (akey, adj_out, lab, kmax, adj_mat, lists)     # adj_mat kept alive so the key cannot be recycled
                self.__dict__["_adj_cache"] = cached
            _, adj_out, lab, k_hint, _, nbr_lists = cached
            adj_mat = adj_out                                                        # layers see the expanded matrix (:428, :448)
            if exists(self.adj_emb):
                labels, label_emb = lab, self.adj_emb.weight

        global_tokens = None
        if exists(self.global_tokens):
            global_tokens = self.global_tokens.to(dev).unsqueeze(0).expand(b, -1, -1)

        coor_changes = [coors]
        for global_attn, egnn in self.layers:
            if exists(global_attn):
                feats, global_tokens = global_attn(feats, global_tokens, mask=mask)
            feats, coors = egnn(feats, coors, edges, mask, adj_mat, _edge_labels=labels, _label_emb=label_emb,
                                _k_hint=k_hint, neighbors=nbr_lists if exists(mask) else None)
            coor_changes.append(coors)

        if out_dev != dev:
            feats, coors = feats.to(out_dev), coors.to(out_dev)
        if return_coor_changes:
            return feats, coors, [c.to(out_dev) for c in coor_changes]
        return feats, coors
