"""Three and four heads on the tcgen05 pair kernels (precision='bf16'), on a B200.  `-m gpu`.

At d in {64, 128} (and d = 32 with four heads) the forward and backward kernel A run once per group of at most two heads, with
the head offset as a kernel argument; kernel C runs once with all heads.  Every case first checks that enf_xattn_dispatch
names the tcgen05 kernels, so that a fall-back to the fp32 kernels cannot pass."""
import types

import pytest
import torch

from oracle import enf_ref as R
from helpers import make_case, rel_err, worst_leaf, Checker, compare, TOL_TC, TOL_TC_LEAF, TOL_TC_SMALL
from test_gpu_grad_x import _run, dx_err

pytestmark = pytest.mark.gpu

# run-to-run spread of one build: the backward accumulates with atomics (README: <= 3e-6 of the largest entry at ns64)
TOL_REPEAT = 1e-5

f32 = lambda t: t.to("cuda", torch.float32).contiguous()


def _cfg(d, H, inv, window=True, num_out=1, latent_dim=16, freq=(0.05, 0.1)):
    return R.EnfConfig(num_in=3 if inv.startswith("ball") else 2, num_hidden=d, num_heads=H, num_out=num_out, latent_dim=latent_dim,
                       invariant_type=inv, embedding_freq_multiplier=freq, use_gaussian_window=window)


def _nef(cfg, **kw):
    import enf_pde_b200 as E
    ns = types.SimpleNamespace(invariant_type=cfg.invariant_type, num_in=cfg.num_in)
    return E.EquivariantCrossAttentionNeF(
        num_hidden=cfg.num_hidden, num_heads=cfg.num_heads, num_layers=0, num_out=cfg.num_out, latent_dim=cfg.latent_dim,
        cross_attn_invariant=E.get_ca_invariant(ns), embedding_freq_multiplier=cfg.embedding_freq_multiplier,
        use_gaussian_window=cfg.use_gaussian_window, precision="bf16", **kw)


def _assert_tc(cfg, B, C, Z):
    from enf_pde_b200 import _lib
    from gpu_helpers import desc_for
    assert _lib.dispatch(desc_for(cfg, B, C, Z, precision=1)) == (True, True)      # the tcgen05 kernels, not a fallback


def _fwd_bwd(cfg, params, x, p, a, sigma, d_out, weights_grad=True, **kw):
    P = R.tree_map(lambda t: f32(t).requires_grad_(weights_grad), params)
    pg, ag = f32(p).requires_grad_(True), f32(a).requires_grad_(True)
    sg = f32(sigma).requires_grad_(True) if cfg.use_gaussian_window else None
    out = _nef(cfg, **kw).apply(P, f32(x), pg, ag, sg)
    out.backward(f32(d_out))
    torch.cuda.synchronize()
    g = {k: v.grad for k, v in R.tree_flatten(P["params"]).items()} if weights_grad else None
    return dict(out=out.detach(), dp=pg.grad, da=ag.grad, ds=None if sg is None else sg.grad, g=g)


# ---- 1. every new (d, H) against the fp64 oracle ---------------------------------------------------------------------------
CASES = [
    # (name, d, H, invariant, window, B, C, Z, polar_grid): ragged multi-tile C, window on and off, five invariant kinds
    # (the latent position grid of ponita / rel_pos / rel_pos_periodic needs a square Z)
    ("d128_h3_rel_pos_periodic", 128, 3, "rel_pos_periodic", True, 2, 300, 16, None),
    ("d128_h4_ponita_nowin", 128, 4, "ponita", False, 2, 300, 16, None),
    ("d128_h4_latitude", 128, 4, "latitude_periodic", True, 2, 300, 18, (6, 3)),
    ("d64_h3_latitude", 64, 3, "latitude_periodic", True, 3, 300, 18, (6, 3)),
    ("d64_h3_rel_pos_nowin", 64, 3, "rel_pos", False, 2, 340, 9, None),
    ("d64_h4_ponita", 64, 4, "ponita", True, 3, 300, 25, None),
    ("d32_h4_ball", 32, 4, "ball", True, 2, 300, 25, None),
    ("d32_h4_rel_pos_periodic_nowin", 32, 4, "rel_pos_periodic", False, 3, 310, 9, None),
]


@pytest.mark.parametrize("case", CASES, ids=lambda c: c[0])
def test_heads_against_oracle(case):
    """decoded field, dp, da, dsigma and every weight leaf: the buckets of the tcgen05 parity tests (TOL_TC at d = 128,
    TOL_TC_SMALL below for the latent gradients; TOL_TC_LEAF per leaf, TOL_TC for the field and over all leaves)."""
    name, d, H, inv, window, B, C, Z, grid = case
    cfg = _cfg(d, H, inv, window)
    data = make_case(cfg, B, C, Z, seed=13, polar_grid=grid)
    _assert_tc(cfg, B, C, Z)
    chk = Checker(cfg, data)
    r = _fwd_bwd(cfg, *data)
    tol = TOL_TC if d == 128 else TOL_TC_SMALL
    errs, worst, ok = compare(chk, r["out"], r["dp"], r["da"], r["ds"], r["g"], tol, TOL_TC_LEAF, use_window=window)
    ok = ok and errs["out"] < TOL_TC
    errs["dtheta_global"] = worst_leaf(r["g"], R.tree_flatten(chk.ref[1]["params"]), floor=1.0)[0]
    print(name, {k: f"{v:.2e}" for k, v in errs.items()}, "worst leaf:", worst, "kink allowance used:", chk.used_allowance)
    assert ok and errs["dtheta_global"] < TOL_TC, (errs, worst)


# ---- 2. dx (ENF_FLAG_GRAD_X): kernel C's GX variant with four side-operand heads -------------------------------------------
@pytest.mark.parametrize("d,H,inv,shared", [(128, 3, "rel_pos_periodic", False), (64, 4, "ponita", False), (32, 4, "ball", False),
                                            (128, 4, "rel_pos_periodic", True)])
def test_heads_dx_against_oracle(d, H, inv, shared):
    cfg = _cfg(d, H, inv)
    data = make_case(cfg, 2, 300, 16, seed=17)
    if shared:
        data = (data[0], data[1][:1].expand(2, -1, -1), *data[2:])
    _assert_tc(cfg, 2, 300, 16)
    r = _run(cfg, *data, precision="bf16", shared=shared)
    tol = TOL_TC if d == 128 else TOL_TC_SMALL
    e = dx_err(cfg, data, r["dx"], tol, shared=shared)
    e_dp = rel_err(r["dp"], R.fwd_bwd(cfg, *data)[2])
    print(d, H, inv, "shared" if shared else "", f"dx {e:.2e}  (dp {e_dp:.2e})")
    assert e < tol, (e, e_dp)


# ---- 3. modes ------------------------------------------------------------------------------------------------------------------
MODE_SHAPES = [(128, 3, "rel_pos_periodic"), (64, 4, "ponita"), (32, 4, "ball")]


@pytest.mark.parametrize("d,H,inv", MODE_SHAPES)
def test_heads_recompute_matches_stash_mode(d, H, inv):
    """ENF_FLAG_RECOMPUTE re-runs every head group's forward per chunk of fields: the field is bit-identical, the gradients
    agree with the stash mode to summation-order noise (as tests/test_gpu_modes.py holds H <= 2)."""
    cfg = _cfg(d, H, inv)
    data = make_case(cfg, 3, 300, 16, seed=19)
    _assert_tc(cfg, 3, 300, 16)
    r0 = _fwd_bwd(cfg, *data)
    r1 = _fwd_bwd(cfg, *data, recompute=True, chunk_fields=2)
    assert torch.equal(r0["out"], r1["out"])
    errs = {k: rel_err(r1[k], r0[k]) for k in ("dp", "da", "ds")}
    errs["dtheta"] = worst_leaf(r1["g"], r0["g"])[0]
    print(d, H, {k: f"{v:.1e}" for k, v in errs.items()})
    assert errs["dp"] < 2e-5 and errs["da"] < 2e-5 and errs["ds"] < 2e-5 and errs["dtheta"] < 2e-4, errs


@pytest.mark.parametrize("d,H,inv", MODE_SHAPES)
def test_heads_forward_only_matches_training_forward(d, H, inv):
    """ENF_FLAG_FORWARD_ONLY (no stash, no logits) and ENF_FLAG_OUT_BF16 give the training forward's field."""
    from enf_pde_b200 import _lib
    from gpu_helpers import desc_for
    cfg = _cfg(d, H, inv, num_out=3)
    params, x, p, a, sigma, d_out = make_case(cfg, 2, 300, 16, seed=23)
    desc = desc_for(cfg, 2, 300, 16, precision=1)
    desc.flags = _lib.FLAG_FORWARD_ONLY
    assert _lib.dispatch(desc) == (True, False)
    train = _fwd_bwd(cfg, params, x, p, a, sigma, d_out)["out"]
    P = R.tree_map(f32, params)
    with torch.no_grad():
        infer = _nef(cfg).apply(P, f32(x), f32(p), f32(a), f32(sigma))
        o16 = _nef(cfg, out_bf16=True).apply(P, f32(x), f32(p), f32(a), f32(sigma))
    assert torch.equal(infer, train)
    assert o16.dtype == torch.bfloat16 and torch.equal(o16, infer.to(torch.bfloat16))


@pytest.mark.parametrize("d,H,inv", MODE_SHAPES)
def test_heads_latents_only_and_repeated_backward(d, H, inv):
    """a latents-only backward (weights frozen: no shared-weight gradient MMAs) gives the latent gradients of a full backward,
    and two full backwards agree within the atomics spread the README states."""
    cfg = _cfg(d, H, inv)
    data = make_case(cfg, 2, 300, 16, seed=29)
    _assert_tc(cfg, 2, 300, 16)
    r0 = _fwd_bwd(cfg, *data)
    r1 = _fwd_bwd(cfg, *data)
    rl = _fwd_bwd(cfg, *data, weights_grad=False)
    lat = {k: rel_err(rl[k], r0[k]) for k in ("dp", "da", "ds")}
    rep = {k: rel_err(r1[k], r0[k]) for k in ("dp", "da", "ds")}
    rep["dtheta"] = worst_leaf(r1["g"], r0["g"], floor=1.0)[0]
    print(d, H, "latents only", {k: f"{v:.1e}" for k, v in lat.items()}, "repeat", {k: f"{v:.1e}" for k, v in rep.items()})
    assert torch.equal(r0["out"], r1["out"]) and torch.equal(r0["out"], rl["out"])
    assert all(v < TOL_REPEAT for v in lat.values()), lat
    assert all(v < TOL_REPEAT for v in rep.values()), rep


# ---- 4. head-offset addressing without the oracle ------------------------------------------------------------------------------
def _duplicate_heads(params, d):
    """heads 2, 3 := heads 0, 1 in every H-blocked weight column of the attention (q, k, v projections and the value
    conditioning's gamma | beta output)."""
    attn = params["params"]["cross_attention_blocks_0"]["attn"]

    def dup(t, halves=1):
        t = t.clone()
        w = t.shape[-1] // halves
        for s in range(halves):
            t[..., s * w + 2 * d:s * w + 4 * d] = t[..., s * w:s * w + 2 * d]
        return t
    for k in ("inv_emb_to_q", "a_to_k", "a_to_v"):
        attn[k] = {n: dup(v) for n, v in attn[k].items()}
    attn["inv_emb_to_v"]["Dense_1"] = {n: dup(v, 2) for n, v in attn["inv_emb_to_v"]["Dense_1"].items()}
    return params


@pytest.mark.parametrize("d", [128, 64, 32])
def test_duplicated_heads_give_equal_nbar(d):
    """with heads 2, 3 copies of heads 0, 1 the second head group computes what the first did: nbar's heads 2, 3 equal heads
    0, 1 bit for bit (each head's chain reads only its own U, b3, kappa, W3 and writes only its own slices)."""
    from enf_pde_b200 import _lib
    from enf_pde_b200.nef import _XAttnFunction
    from gpu_helpers import ws_view
    cfg = _cfg(d, 4, "rel_pos_periodic")
    params, x, p, a, sigma, d_out = make_case(cfg, 2, 300, 16, seed=31)
    params = _duplicate_heads(params, d)
    _assert_tc(cfg, 2, 300, 16)
    P = R.tree_map(f32, params)
    out = _nef(cfg).apply(P, f32(x), f32(p).requires_grad_(True), f32(a), f32(sigma))     # the autograd node keeps the workspace
    torch.cuda.synchronize()
    desc_kw, ws_ref, _ = _XAttnFunction.last_ws
    nbar = ws_view(_lib.load(), _lib.EnfDesc(**desc_kw), ws_ref(), "nbar").view(2, 300, 4, d)
    lse = ws_view(_lib.load(), _lib.EnfDesc(**desc_kw), ws_ref(), "lse").view(2, 300, 4)
    assert out.shape == (2, 300, 1)
    print(d, "max |nbar[2:] - nbar[:2]|", float((nbar[:, :, 2:] - nbar[:, :, :2]).abs().max()))
    assert torch.equal(nbar[:, :, 2:], nbar[:, :, :2]) and torch.equal(lse[:, :, 2:], lse[:, :, :2])
    assert not torch.equal(nbar[:, :, 1], nbar[:, :, 0])


# ---- 5. full size -----------------------------------------------------------------------------------------------------------------
def test_heads_full_size_ns_subset():
    """BASELINE config 2's shape (B = 32, C = 4096, Z = 64, d = 128) at H = 3, forward and backward on the tcgen05 kernels,
    against the fp32 kernels on a cotangent supported on a subset of rows (queries are independent)."""
    import enf_pde_b200 as E
    cfg = _cfg(128, 3, "rel_pos_periodic")
    B, C, Z = 32, 4096, 64
    params, _, p, a, sigma, _ = make_case(cfg, B, 8, Z, seed=7)
    x = R.make_coords(cfg, (64, 64)).float().double()[None].expand(B, -1, -1)
    g = torch.Generator().manual_seed(11)
    sub = torch.randperm(C, generator=g)[:24]
    d_out = torch.zeros(B, C, 1, dtype=torch.float64)
    d_out[:, sub] = torch.randn(B, 24, 1, generator=g, dtype=torch.float64)
    _assert_tc(cfg, B, C, Z)
    tc = _fwd_bwd(cfg, params, x, p, a, sigma, d_out)
    ns = types.SimpleNamespace(invariant_type=cfg.invariant_type, num_in=cfg.num_in)
    ref_nef = E.EquivariantCrossAttentionNeF(num_hidden=128, num_heads=3, num_layers=0, num_out=1, latent_dim=16,
                                             cross_attn_invariant=E.get_ca_invariant(ns),
                                             embedding_freq_multiplier=cfg.embedding_freq_multiplier, precision="fp32")
    P = R.tree_map(lambda t: f32(t).requires_grad_(True), params)
    pg, ag, sg = (f32(t).requires_grad_(True) for t in (p, a, sigma))
    out = ref_nef.apply(P, f32(x), pg, ag, sg)
    out.backward(f32(d_out))
    bsel = [0, 13, 31]
    errs = dict(out=rel_err(tc["out"][bsel][:, sub], out.detach()[bsel][:, sub]), dp=rel_err(tc["dp"][bsel], pg.grad[bsel]),
                da=rel_err(tc["da"][bsel], ag.grad[bsel]), ds=rel_err(tc["ds"][bsel], sg.grad[bsel]))
    print("full-size H = 3 tc vs fp32 kernels", {k: f"{v:.2e}" for k, v in errs.items()})
    assert all(v < TOL_TC for v in errs.values()), errs
