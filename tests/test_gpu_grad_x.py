"""Gradient w.r.t. the query coordinates x (ENF_FLAG_GRAD_X, enf_xattn_bwd_x) on a B200, through nef.apply + autograd:
fp32 and tcgen05 backward against the oracle's fp64 autograd, an oracle-free translation identity, and the guarantee that
asking for dx changes nothing else.  `-m gpu`."""
import types

import pytest
import torch

from oracle import enf_ref as R
from helpers import golden_names, load_golden, make_case, rel_err, worst_leaf, TOL_FP32, TOL_TC, TOL_TC_SMALL

pytestmark = pytest.mark.gpu

# run-to-run spread of one build: the backward accumulates with atomics (README: <= 3e-6 of the largest entry at ns64)
TOL_REPEAT = 1e-5


def _nef(cfg, precision="fp32", recompute=False):
    import enf_pde_b200 as E
    ns = types.SimpleNamespace(invariant_type=cfg.invariant_type, num_in=cfg.num_in)
    return E.EquivariantCrossAttentionNeF(
        num_hidden=cfg.num_hidden, num_heads=cfg.num_heads, num_layers=cfg.num_layers, num_out=cfg.num_out,
        latent_dim=cfg.latent_dim, cross_attn_invariant=E.get_ca_invariant(ns), self_attn_invariant=E.get_sa_invariant(ns),
        embedding_freq_multiplier=cfg.embedding_freq_multiplier, use_gaussian_window=cfg.use_gaussian_window,
        precision=precision, recompute=recompute, chunk_fields=2 if recompute else 0)


def _run(cfg, params, x, p, a, sigma, d_out, precision="fp32", grad_x=True, shared=False, recompute=False):
    """fwd + bwd through nef.apply; x (B,C,Dx), or with shared=True ONE grid x[0] (C,Dx) for every field."""
    f = lambda t: t.to("cuda", torch.float32).contiguous()
    P = R.tree_map(lambda t: f(t).requires_grad_(True), params)
    xg = f(x[0] if shared else x).requires_grad_(grad_x)
    pg, ag = f(p).requires_grad_(True), f(a).requires_grad_(True)
    sg = f(sigma).requires_grad_(True) if cfg.use_gaussian_window else None
    out = _nef(cfg, precision, recompute).apply(P, xg, pg, ag, sg)
    out.backward(f(d_out))
    torch.cuda.synchronize()
    return dict(out=out.detach(), dx=xg.grad, dp=pg.grad, da=ag.grad, ds=None if sg is None else sg.grad,
                g=R.tree_flatten(R.tree_map(lambda t: t.grad, P)["params"]))


def oracle_dx(cfg, params, x, p, a, sigma, d_out, shared=False, kink=0.0):
    """fp64 autograd of <d_out, nef_apply> w.r.t. x (shared: w.r.t. the one grid, i.e. summed over fields).  kink: the relu
    derivative's threshold (helpers.kink_allowance)."""
    xg = (x[0] if shared else x).detach().clone().requires_grad_(True)
    R.RELU_KINK_SHIFT[0] = kink
    try:
        out = R.nef_apply(cfg, params, xg.expand(x.shape) if shared else xg, p, a, sigma)
        (dx,) = torch.autograd.grad(out, xg, grad_outputs=d_out)
    finally:
        R.RELU_KINK_SHIFT[0] = 0.0
    return dx


def dx_err(cfg, case, got, tol, shared=False, tau=4e-6):
    """rel_err of dx against the oracle; over `tol`, with the relu-kink allowance of helpers.kink_allowance subtracted."""
    want = oracle_dx(cfg, *case, shared=shared)
    e = rel_err(got, want)
    if e < tol:
        return e
    allow = sum((oracle_dx(cfg, *case, shared=shared, kink=s) - want).abs() for s in (tau, -tau))
    e2 = ((got.double().cpu() - want).abs() - allow).clamp(min=0).max().item() / want.abs().max().item()
    return min(e, e2)


# ---- 1. fp32 parity on every golden fixture ------------------------------------------------------------------------------
@pytest.mark.parametrize("name", golden_names() + golden_names(sa=True))
def test_fp32_dx_on_golden_fixtures(name):
    cfg, params, _, rec = load_golden(name)
    case = (params, rec["x"], rec["p"], rec["a"], rec["sigma"], rec["cot"])
    r = _run(cfg, *case)
    e = dx_err(cfg, case, r["dx"], TOL_FP32)
    print(name, f"dx {e:.2e}")
    assert r["dx"].shape == rec["x"].shape and e < TOL_FP32, e


@pytest.mark.parametrize("inv,layers", [("rel_pos_periodic", 0), ("ponita", 0), ("latitude_periodic", 0), ("ball", 0),
                                        ("rel_pos_periodic", 1)])
def test_fp32_dx_shared_grid(inv, layers):
    """one 2-D grid for all fields (x_batch_stride = 0): dx is [C,Dx], the sum over fields."""
    grid = (6, 3) if inv == "latitude_periodic" else None
    cfg = R.EnfConfig(num_in=3 if inv == "ball" else 2, num_hidden=32, num_heads=2, num_out=2, latent_dim=8, invariant_type=inv,
                      embedding_freq_multiplier=(0.1, 0.2), num_layers=layers)
    params, x, p, a, sigma, d_out = make_case(cfg, 3, 70, 18 if grid else 9, seed=21, polar_grid=grid)
    x = x[:1].expand(3, -1, -1)
    case = (params, x, p, a, sigma, d_out)
    r = _run(cfg, *case, shared=True)
    e = dx_err(cfg, case, r["dx"], TOL_FP32, shared=True)
    print(inv, layers, f"dx {e:.2e}")
    assert r["dx"].shape == x.shape[1:] and e < TOL_FP32, e


# ---- 2. tensor-core parity (the shapes of the tcgen05 parity cases of test_gpu_parity.py) ---------------------------------
TC_CASES = [
    # (name, cfg kwargs, B, C, Z, polar_grid, seed)
    ("ns_d128", dict(num_in=2, num_hidden=128, num_heads=2, num_out=1, latent_dim=16, invariant_type="rel_pos_periodic",
                     embedding_freq_multiplier=(0.05, 0.1)), 2, 75, 16, None, 3),
    ("plane_d64", dict(num_in=2, num_hidden=64, num_heads=2, num_out=1, latent_dim=16, invariant_type="ponita",
                       embedding_freq_multiplier=(0.05, 0.01)), 3, 100, 25, None, 3),
    ("sw_d128", dict(num_in=2, num_hidden=128, num_heads=2, num_out=3, latent_dim=32, invariant_type="latitude_periodic",
                     embedding_freq_multiplier=(0.05, 0.2)), 1, 90, 18, (6, 3), 3),
    ("ihc_d32_h3", dict(num_in=3, num_hidden=32, num_heads=3, num_out=1, latent_dim=32, invariant_type="ball",
                        embedding_freq_multiplier=(0.2, 0.5)), 2, 200, 40, None, 3),
    ("tc_multi_tile", dict(num_in=2, num_hidden=128, num_heads=2, num_out=1, latent_dim=16, invariant_type="rel_pos_periodic",
                           embedding_freq_multiplier=(0.05, 0.1)), 5, 300, 36, None, 5),
    ("tc_one_head", dict(num_in=2, num_hidden=128, num_heads=1, num_out=2, latent_dim=8, invariant_type="ponita",
                         embedding_freq_multiplier=(0.05, 0.05)), 2, 200, 9, None, 5),
    ("tc_sphere_window", dict(num_in=2, num_hidden=128, num_heads=2, num_out=3, latent_dim=32, invariant_type="latitude_periodic",
                              embedding_freq_multiplier=(0.05, 0.2)), 2, 260, 18, (6, 3), 5),
    ("tc_one_query", dict(num_in=2, num_hidden=128, num_heads=2, num_out=1, latent_dim=16, invariant_type="rel_pos_periodic",
                          embedding_freq_multiplier=(0.05, 0.1)), 2, 1, 16, None, 7),
    ("tc_one_latent", dict(num_in=2, num_hidden=64, num_heads=1, num_out=1, latent_dim=16, invariant_type="ponita",
                           embedding_freq_multiplier=(0.05, 0.05)), 2, 150, 1, None, 7),
]


@pytest.mark.parametrize("case", TC_CASES, ids=lambda c: c[0])
def test_tensor_core_dx_against_oracle(case):
    """kernel C's GX variant: dx held to the bucket the tcgen05 parity tests apply to dp on the same shape (TOL_TC at d = 128,
    TOL_TC_SMALL below); dp is checked beside it as the reference point."""
    from enf_pde_b200 import _lib
    from gpu_helpers import desc_for
    name, kw, B, C, Z, grid, seed = case
    cfg = R.EnfConfig(**kw)
    data = make_case(cfg, B, C, Z, seed=seed, polar_grid=grid)
    assert _lib.dispatch(desc_for(cfg, B, C, Z, precision=1)) == (True, True)      # the tcgen05 kernels, not a fallback
    r = _run(cfg, *data, precision="bf16")
    tol = TOL_TC if cfg.num_hidden == 128 else TOL_TC_SMALL
    e = dx_err(cfg, data, r["dx"], tol)
    e_dp = rel_err(r["dp"], R.fwd_bwd(cfg, *data)[2])
    print(name, f"dx {e:.2e}  (dp {e_dp:.2e})")
    assert e < tol, (e, e_dp)


# ---- 3. translation identity (no oracle) ----------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("inv", ["rel_pos", "rel_pos_periodic", "ponita"])
def test_translation_identity(inv, precision):
    """out depends on x and the latent positions only through their difference, so per field
    sum_c dx[c] + sum_z dp[z, :n_pos] = 0: ties the new gradient to the existing dp."""
    cfg = R.EnfConfig(num_in=2, num_hidden=128 if precision == "bf16" else 32, num_heads=2, num_out=1, latent_dim=16,
                      invariant_type=inv, embedding_freq_multiplier=(0.05, 0.1))
    params, x, p, a, sigma, d_out = make_case(cfg, 3, 300, 25, seed=31)
    r = _run(cfg, params, x, p, a, sigma, d_out, precision=precision)
    sx = r["dx"].double().sum(1)
    sp = r["dp"].double()[:, :, :2].sum(1)
    e = float((sx + sp).abs().max() / sp.abs().max())
    print(inv, precision, f"identity {e:.2e}", f"max|sum dp| {float(sp.abs().max()):.3e}")
    assert e < (TOL_FP32 if precision == "fp32" else TOL_TC), e


# ---- 4. nothing else changes ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision,d", [("fp32", 32), ("bf16", 128), ("bf16", 64), ("bf16", 32)])
def test_grad_x_changes_nothing_else(precision, d):
    """with ENF_FLAG_GRAD_X: bit-identical field, every other gradient within the atomics spread of repeated runs (weight
    gradients against the largest entry over all leaves, as the README states that spread); ENF_FLAG_RECOMPUTE gives the stash
    mode's dx."""
    H = 3 if d == 32 and precision == "bf16" else 2
    inv = "ball" if H == 3 else "rel_pos_periodic"
    cfg = R.EnfConfig(num_in=3 if inv == "ball" else 2, num_hidden=d, num_heads=H, num_out=1, latent_dim=16, invariant_type=inv,
                      embedding_freq_multiplier=(0.05, 0.1))
    data = make_case(cfg, 5, 300, 25, seed=41)
    r0 = _run(cfg, *data, precision=precision, grad_x=False)
    r1 = _run(cfg, *data, precision=precision, grad_x=True)
    assert r0["dx"] is None and r1["dx"] is not None
    assert torch.equal(r0["out"], r1["out"])
    errs = {k: rel_err(r1[k], r0[k]) for k in ("dp", "da", "ds")}
    errs["dtheta"] = worst_leaf(r1["g"], r0["g"], floor=1.0)[0]
    rr = _run(cfg, *data, precision=precision, grad_x=False)          # the spread of two runs without the flag, for the log
    spread = {k: rel_err(rr[k], r0[k]) for k in ("dp", "da", "ds")}
    spread["dtheta"] = worst_leaf(rr["g"], r0["g"], floor=1.0)[0]
    print(precision, d, "with vs without dx", {k: f"{v:.1e}" for k, v in errs.items()},
          "two runs without", {k: f"{v:.1e}" for k, v in spread.items()})
    assert all(v < TOL_REPEAT for v in errs.values()), errs
    if precision == "bf16":
        rr = _run(cfg, *data, precision=precision, recompute=True)
        e = rel_err(rr["dx"], r1["dx"])
        print("recompute dx", f"{e:.1e}")
        assert torch.equal(rr["out"], r1["out"]) and e < TOL_REPEAT, e


# ---- 5. autograd wiring ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_autograd_wiring(precision):
    from enf_pde_b200 import _lib
    from enf_pde_b200.nef import _XAttnFunction
    cfg = R.EnfConfig(num_in=2, num_hidden=128, num_heads=2, num_out=1, latent_dim=16, invariant_type="rel_pos_periodic",
                      embedding_freq_multiplier=(0.05, 0.1))
    params, x, p, a, sigma, d_out = make_case(cfg, 2, 150, 16, seed=51)
    f = lambda t: t.to("cuda", torch.float32)
    nef = _nef(cfg, precision)
    P = R.tree_map(f, params)                                         # nothing but x requires grad
    want = oracle_dx(cfg, params, x, p, a, sigma, d_out)
    tol = TOL_FP32 if precision == "fp32" else TOL_TC
    # x as the only input that requires grad (was: the forward-only path, then ENF_ERR_STATE); torch.autograd.grad
    xg = f(x).requires_grad_(True)
    out = nef.apply(P, xg, f(p), f(a), f(sigma))
    assert _XAttnFunction.last_ws[0]["flags"] == _lib.FLAG_GRAD_X
    (dx,) = torch.autograd.grad(out, xg, grad_outputs=f(d_out))
    assert rel_err(dx, want) < tol
    # a coordinate map x = theta[0] * x0 + theta[1] delivers its gradient to theta
    theta = torch.tensor([1.25, 0.1], device="cuda", requires_grad=True)
    x0 = (x - 0.1) / 1.25
    out = nef.apply(P, theta[0] * f(x0) + theta[1], f(p), f(a), f(sigma))
    out.backward(f(d_out))
    want_theta = torch.stack([(want * x0).sum(), want.sum()])
    e = float((theta.grad.double().cpu() - want_theta).abs().max() / want_theta.abs().max())
    print(precision, "theta", theta.grad.tolist(), want_theta.tolist(), f"{e:.1e}")
    assert e < tol, e
    # without x requiring grad nothing changes: no flag, same workspace as before
    with torch.no_grad():
        nef.apply(P, f(x), f(p), f(a), f(sigma))
    assert _XAttnFunction.last_ws[0]["flags"] == _lib.FLAG_FORWARD_ONLY
