"""Helpers shared by the GPU parity tests, smoke() and bench.py: build the product modules from
a tests/cases.py case and move numpy inputs to torch."""
from __future__ import annotations

import numpy as np
import torch

import cases


def to_torch(x, dtype, device):
    if x is None:
        return None
    x = np.asarray(x)
    if x.dtype == bool:
        return torch.from_numpy(x.copy()).to(device)
    if np.issubdtype(x.dtype, np.integer):
        return torch.from_numpy(x.astype(np.int64)).to(device)
    return torch.from_numpy(x.astype(np.float64)).to(device=device, dtype=dtype)


def make_module(case, dtype, device="cuda", **extra):
    from egnn_pytorch_b200 import EGNN, EGNN_Network
    spec = case["spec"]
    mod = EGNN_Network(**spec["cfg"], **extra) if case["kind"] == "network" else EGNN(**spec["cfg"], **extra)
    mod = mod.to(dtype)                            # before loading: load_state_dict casts to the parameter dtype
    sd = {k: torch.from_numpy(np.asarray(v, dtype=np.float64)) for k, v in case["params"].items()}
    mod.load_state_dict(sd, strict=True)          # reference state-dict keys must load unchanged
    return mod.to(device).eval()


def run_module(mod, case, dtype, device="cuda", **kw):
    ins = case["inputs"]
    t = lambda name: to_torch(ins.get(name), dtype, device)
    if case["kind"] == "network":
        return mod(t("feats"), t("coors"), adj_mat=t("adj_mat"), edges=t("edges"), mask=t("mask"), **kw)
    return mod(t("feats"), t("coors"), t("edges"), mask=t("mask"), adj_mat=t("adj_mat"), **kw)


def module_grads(case, dtype, device="cuda", **kw):
    """Run forward + backward of the product module; -> flat {name: float64 numpy gradient}.  Extra keyword arguments
    (e.g. `neighbors=`) go to the module call."""
    mod = make_module(case, dtype, device=device)
    mod.requires_grad_(True)
    ins = case["inputs"]
    t = lambda name: to_torch(ins.get(name), dtype, device)
    feats, coors, edges = t("feats"), t("coors"), t("edges")
    leaves = {"coors": coors.requires_grad_(True)}
    if feats.is_floating_point():
        leaves["feats"] = feats.requires_grad_(True)
    if edges is not None and edges.is_floating_point():
        leaves["edges"] = edges.requires_grad_(True)
    gf, gx = (torch.from_numpy(g).to(device=device, dtype=dtype) for g in cases.upstream_grads(case))
    with torch.enable_grad():
        if case["kind"] == "network":
            fo, xo = mod(feats, coors, adj_mat=t("adj_mat"), edges=edges, mask=t("mask"), **kw)
        else:
            fo, xo = mod(feats, coors, edges, mask=t("mask"), adj_mat=t("adj_mat"), **kw)
        assert fo.requires_grad and xo.requires_grad
        ((fo * gf).sum() + (xo * gx).sum()).backward()
    out = {f"in.{k}": v.grad.double().cpu().numpy() for k, v in leaves.items()}
    for k, p in mod.named_parameters():
        out[f"p.{k}"] = (torch.zeros_like(p) if p.grad is None else p.grad).double().cpu().numpy()
    return out


def compare(got, want, tol, what):
    """Every gradient tensor within `tol` of max(1, max|want|)."""
    assert set(got) == set(want), (what, sorted(set(got) ^ set(want)))
    bad = []
    for k in sorted(want):
        scale = max(1.0, float(np.abs(want[k]).max()))
        err = float(np.abs(got[k] - want[k]).max()) / scale
        if not np.isfinite(got[k]).all() or err > tol:
            bad.append(f"{k}: rel err {err:.3e}")
    assert not bad, f"{what}: " + "; ".join(bad)


def grad_tol(case, dtype):
    if dtype == torch.float64:
        # CoorsNorm: the oracle (like the reference) carries ~1e-9 of cancellation noise from the 1/eps self pair
        return 1e-7 if "norm_coors" in str(case["spec"]["cfg"]) else 1e-9
    return 5e-4


def max_err(a, b):
    a = a.detach().double().cpu().numpy() if torch.is_tensor(a) else np.asarray(a, np.float64)
    b = b.detach().double().cpu().numpy() if torch.is_tensor(b) else np.asarray(b, np.float64)
    return float(np.abs(a - b).max())


def assert_close(got, want, atol, rtol, what=""):
    got = got.detach().double().cpu().numpy() if torch.is_tensor(got) else np.asarray(got, np.float64)
    want = np.asarray(want, np.float64)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    assert np.isfinite(got).all(), f"{what}: non-finite output"
    err = np.abs(got - want)
    tol = atol + rtol * np.abs(want)
    worst = float((err - tol).max())
    assert worst <= 0, f"{what}: max|err|={err.max():.3e} exceeds atol={atol} rtol={rtol} (|want|max={np.abs(want).max():.3e})"
