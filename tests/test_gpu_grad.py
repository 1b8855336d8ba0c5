"""Backward parity on the GPU: gradients of the CUDA modules (torch.autograd.Function over egnn_layer_backward)
against the numpy backward oracle and against the committed gradients of the reference's own autograd
(tests/golden/grad_*.npz), for the same loss  sum(feats_out * G_f) + sum(coors_out * G_x)."""
import os

import numpy as np
import pytest
import torch

import cases
import util

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _grad_dtype(name):
    # m_dim = 32 in fp64 exceeds the shared-memory budget of the first backward kernel (EGNN_ERR_UNSUPPORTED)
    return torch.float32 if name == "dense_mdim32" else torch.float64


GRAD_CASES = cases.GRAD_SPECS + ["c1_dim512_xavier"]


@pytest.mark.parametrize("name", GRAD_CASES)
def test_grads_match_oracle_fp64(name):
    case = cases.build_case(cases.SPECS[name])
    dtype = _grad_dtype(name)
    got = util.module_grads(case, dtype)
    want = cases.flatten_grads(cases.run_oracle_grad(case))
    util.compare(got, want, util.grad_tol(case, dtype), f"{name} vs oracle")


@pytest.mark.parametrize("name", cases.GRAD_SPECS)
def test_grads_match_reference_fixture_fp64(name):
    g = np.load(os.path.join(GOLDEN, f"grad_{name}.npz"))
    if bool(g["tie_dependent"]):
        pytest.skip("reference gradients depend on torch.topk's tie order")
    case = cases.build_case(cases.SPECS[name])
    assert cases.case_checksum(case) == str(g["checksum"])
    dtype = _grad_dtype(name)
    got = util.module_grads(case, dtype)
    want = {k: g[k] for k in g.files if k.startswith(("in.", "p."))}
    util.compare(got, want, util.grad_tol(case, dtype), f"{name} vs reference autograd")


@pytest.mark.parametrize("name", ["dense_xavier", "dense_everything", "knn_edges_mask", "adj_sparse_random",
                                  "net_c3_xavier", "net_c5_xavier", "dense_mdim32"])
def test_grads_fp32(name):
    case = cases.build_case(cases.SPECS[name])
    got = util.module_grads(case, torch.float32)
    want = cases.flatten_grads(cases.run_oracle_grad(case))
    util.compare(got, want, util.grad_tol(case, torch.float32), f"{name} fp32 vs oracle")


@pytest.mark.parametrize("name", ["dense_everything", "dense_edges", "c1_dim512_xavier", "net_dense_feats", "knn_edges_mask",
                                  "net_c5_xavier"])
def test_grads_with_recompute_instead_of_saved_pair_activations(name, monkeypatch):
    """Dense training keeps 64 B per pair by default (EgnnLayerIO.pre2_out); with the budget set to 0 the backward
    recomputes them with the register-tiled forward kernel -- both routes must give the same gradients."""
    monkeypatch.setenv("EGNN_B200_SAVE_PAIR_MB", "0")
    case = cases.build_case(cases.SPECS[name])
    got = util.module_grads(case, torch.float64)
    want = cases.flatten_grads(cases.run_oracle_grad(case))
    util.compare(got, want, util.grad_tol(case, torch.float64), f"{name} (recompute) vs oracle")


def test_cpu_tensors_and_bf16_modules_train_through_the_gpu_kernels():
    """CPU fp64 tensors (how the reference's tests call the layer) get CPU gradients; a bf16 module trains through
    the fp32 kernels and returns bf16 gradients."""
    case = cases.build_case(cases.SPECS["dense_edges"])
    got = util.module_grads(case, torch.float64, device="cpu")
    want = cases.flatten_grads(cases.run_oracle_grad(case))
    util.compare(got, want, 1e-9, "cpu staging")
    mod = util.make_module(case, torch.bfloat16).requires_grad_(True)
    ins = case["inputs"]
    f = util.to_torch(ins["feats"], torch.bfloat16, "cuda").requires_grad_(True)
    x = util.to_torch(ins["coors"], torch.float32, "cuda").requires_grad_(True)
    e = util.to_torch(ins["edges"], torch.bfloat16, "cuda")
    with torch.enable_grad():
        fo, xo = mod(f, x, e)
        (fo.float().sum() + xo.sum()).backward()
    assert mod.last_path == "fp32-simt"
    assert f.grad.dtype == torch.bfloat16 and x.grad.dtype == torch.float32
    assert mod.edge_mlp[0].weight.grad.dtype == torch.bfloat16
    assert torch.isfinite(f.grad.float()).all() and torch.isfinite(x.grad).all()


def test_no_graph_is_kept_without_grad():
    case = cases.build_case(cases.SPECS["dense_basic"])
    mod = util.make_module(case, torch.float32).requires_grad_(True)
    out = util.run_module(mod, case, torch.float32)          # autouse fixture: grad mode off
    assert not out[0].requires_grad and out[0].grad_fn is None


def test_training_steps_reduce_the_loss():
    """The reference's denoising loop (denoise_sparse.py:70-78) in miniature: Adam on an EGNN_Network."""
    from egnn_pytorch_b200 import EGNN_Network
    torch.manual_seed(0)
    net = EGNN_Network(num_tokens=21, dim=16, depth=2, num_nearest_neighbors=6, norm_coors=True,
                       coor_weights_clamp_value=2.0).cuda()
    opt = torch.optim.Adam(net.parameters(), lr=1e-2)
    tokens = torch.randint(0, 21, (2, 32), device="cuda")
    coors = torch.randn(2, 32, 3, device="cuda")
    noised = coors + 0.3 * torch.randn_like(coors)
    losses = []
    with torch.enable_grad():
        for _ in range(40):
            _, denoised = net(tokens, noised)
            loss = ((denoised - coors) ** 2).mean()
            opt.zero_grad()
            loss.backward()
            opt.step()
            losses.append(float(loss.detach()))
    assert np.isfinite(losses).all()
    assert losses[-1] < 0.95 * losses[0], losses


def test_backward_c2_shape_runs_and_matches_directional_derivative():
    """Full BASELINE size (dim=512, N=1024, B=1 to bound the time): the analytic gradient along a random direction
    against a central difference of the CUDA forward itself (fp64)."""
    from egnn_pytorch_b200 import EGNN
    torch.manual_seed(1)
    mod = EGNN(dim=512).double().cuda()
    feats = torch.randn(1, 1024, 512, device="cuda", dtype=torch.float64)
    coors = torch.randn(1, 1024, 3, device="cuda", dtype=torch.float64)
    gf, gx = torch.randn_like(feats), torch.randn_like(coors)
    loss = lambda f, x: float(((lambda o: (o[0] * gf).sum() + (o[1] * gx).sum())(mod(f, x))))
    fr, xr = feats.clone().requires_grad_(True), coors.clone().requires_grad_(True)
    with torch.enable_grad():
        fo, xo = mod(fr, xr)
        ((fo * gf).sum() + (xo * gx).sum()).backward()
    vf, vx = torch.randn_like(feats), torch.randn_like(coors)
    eps = 1e-5
    fd = (loss(feats + eps * vf, coors + eps * vx) - loss(feats - eps * vf, coors - eps * vx)) / (2 * eps)
    an = float((fr.grad * vf).sum() + (xr.grad * vx).sum())
    assert abs(fd - an) <= 1e-5 * max(1.0, abs(an)), (fd, an)
    w = mod.edge_mlp[0].weight
    vw = torch.randn_like(w)
    with torch.no_grad():
        w.add_(eps * vw); hi = loss(feats, coors)
        w.sub_(2 * eps * vw); lo = loss(feats, coors)
        w.add_(eps * vw)
    fdw = (hi - lo) / (2 * eps)
    anw = float((w.grad * vw).sum())
    assert abs(fdw - anw) <= 1e-5 * max(1.0, abs(anw)), (fdw, anw)


def test_edge_list_mode_with_empty_slots_matches_directional_derivative():
    """`neighbors=` lists with -1 (empty) slots: analytic gradients along a random direction against a central
    difference of the CUDA forward itself (fp64)."""
    from egnn_pytorch_b200 import EGNN
    torch.manual_seed(3)
    B, N, d, k = 2, 24, 16, 6
    mod = EGNN(dim=d, edge_dim=2, norm_coors=True, m_pool_method="mean").double().cuda()
    for p in mod.parameters():                      # the reference's 1e-3 init hides errors: use O(1) weights
        if p.dim() == 2:
            torch.nn.init.xavier_normal_(p)
    feats = torch.randn(B, N, d, device="cuda", dtype=torch.float64)
    coors = torch.randn(B, N, 3, device="cuda", dtype=torch.float64)
    edges = torch.randn(B, N, N, 2, device="cuda", dtype=torch.float64)
    mask = torch.ones(B, N, dtype=torch.bool, device="cuda")
    mask[1, -3:] = False
    nbrs = torch.stack([torch.stack([torch.randperm(N)[:k] for _ in range(N)]) for _ in range(B)]).int().cuda()
    nbrs[:, ::3, -2:] = -1                          # every third node has two empty slots
    nbrs[0, 5, :] = -1                              # and one node has no neighbours at all
    gf, gx = torch.randn_like(feats), torch.randn_like(coors)

    def loss(f, x, e):
        fo, xo = mod(f, x, e, mask=mask, neighbors=nbrs)
        return (fo * gf).sum() + (xo * gx).sum()

    fr, xr, er = (t.clone().requires_grad_(True) for t in (feats, coors, edges))
    with torch.enable_grad():
        loss(fr, xr, er).backward()
    vf, vx, ve = torch.randn_like(feats), torch.randn_like(coors), torch.randn_like(edges)
    eps = 1e-6
    fd = float(loss(feats + eps * vf, coors + eps * vx, edges + eps * ve) -
               loss(feats - eps * vf, coors - eps * vx, edges - eps * ve)) / (2 * eps)
    an = float((fr.grad * vf).sum() + (xr.grad * vx).sum() + (er.grad * ve).sum())
    assert np.isfinite(an) and abs(fd - an) <= 1e-6 * max(1.0, abs(an)), (fd, an)
    for p in mod.parameters():
        assert torch.isfinite(p.grad).all()


def test_second_backward_and_inplace_edits_are_reported():
    """ADVICE r1: the saved state aliases inputs / parameters -- a second backward or an in-place edit between forward and
    backward must raise, not silently differentiate stale data."""
    from egnn_pytorch_b200 import EGNN
    torch.manual_seed(0)
    mod = EGNN(dim=16).cuda()
    f = torch.randn(1, 12, 16, device="cuda", requires_grad=True)
    x = torch.randn(1, 12, 3, device="cuda", requires_grad=True)
    with torch.enable_grad():
        fo, xo = mod(f, x)
        loss = fo.sum() + xo.sum()
        loss.backward(retain_graph=True)
        with pytest.raises(RuntimeError, match="second time"):
            loss.backward()
        fo, xo = mod(f, x)
        with torch.no_grad():
            mod.edge_mlp[0].weight.mul_(1.5)            # e.g. an optimizer step before backward
        with pytest.raises(RuntimeError, match="modified in place"):
            (fo.sum() + xo.sum()).backward()
