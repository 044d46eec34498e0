"""Gradient w.r.t. the query coordinates (ENF_FLAG_GRAD_X, enf_xattn_bwd_x): the C ABI's host side and the fp64 reference
the GPU tests compare against.  CPU only."""
import ctypes
import os
import re

import pytest
import torch

import enf_pde_b200 as E
from enf_pde_b200 import _lib
from oracle import enf_ref as R
from helpers import golden_names, load_golden, rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OK = dict(B=3, C=70, Z=9, d=32, H=2, L=8, O=1, Dx=2, invariant_kind=3, use_window=1, precision=0, flags=0)


def _bytes(**kw):
    return _lib.load().enf_xattn_workspace_bytes(ctypes.byref(_lib.EnfDesc(**{**OK, **kw})))


def test_grad_x_is_declared_and_exported():
    header = open(os.path.join(ROOT, "include", "enf_b200.h")).read()
    assert re.search(r"int enf_xattn_bwd_x\s*\(", header)
    assert "ENF_FLAG_GRAD_X = 128" in header and _lib.FLAG_GRAD_X == 128
    assert "enf_xattn_bwd_x" in _lib.EXPORTS
    assert hasattr(E.load_library(), "enf_xattn_bwd_x")


def test_grad_x_flag_validation():
    lib = _lib.load()
    assert _bytes(flags=_lib.FLAG_GRAD_X) > 0
    assert _bytes(flags=_lib.FLAG_GRAD_X | _lib.FLAG_RECOMPUTE, precision=1, d=128) > 0
    # no backward, or a self-attention step (x is ignored there; dp carries the poses in both roles)
    selfblk = dict(C=9, O=32, flags=_lib.FLAG_SELF_BLOCK)
    assert _bytes(**selfblk) > 0
    for bad in (dict(flags=_lib.FLAG_GRAD_X | _lib.FLAG_FORWARD_ONLY), dict(selfblk, flags=_lib.FLAG_SELF_BLOCK | _lib.FLAG_GRAD_X)):
        assert _bytes(**bad) == 0, bad
        assert b"ENF_FLAG_GRAD_X" in lib.enf_last_error()


@pytest.mark.parametrize("precision,d,extra", [(0, 32, 0), (1, 128, 0), (1, 128, _lib.FLAG_RECOMPUTE), (1, 64, 0)])
def test_workspace_grows_by_exactly_the_record_cotangents(precision, d, extra):
    lib = _lib.load()
    base = dict(precision=precision, d=d, flags=extra)
    n0, n1 = _bytes(**base), _bytes(**{**base, "flags": extra | _lib.FLAG_GRAD_X})
    B, C = OK["B"], OK["C"]
    assert n0 > 0 and n1 - n0 == ((B * C * 8 + 63) // 64 * 64) * 4      # g_xi [B,C,8], 256-byte granularity
    desc = _lib.EnfDesc(**{**OK, **base, "flags": extra | _lib.FLAG_GRAD_X})
    n = ctypes.c_int64(0)
    assert lib.enf_debug_ws_offset(ctypes.byref(desc), b"g_xi", ctypes.byref(n)) > 0 and n.value == B * C * 8
    assert lib.enf_debug_ws_offset(ctypes.byref(_lib.EnfDesc(**{**OK, **base})), b"g_xi", None) == -1


def test_bwd_x_argument_checks_without_a_gpu():
    """dx without ENF_FLAG_GRAD_X is a state error; a GRAD_X description needs dx (checked before any device work)."""
    lib = _lib.load()
    w = _lib.EnfWeights(**{n: 16 for n in _lib.LEAVES})
    for flags, dx, want in ((0, 256, -7), (_lib.FLAG_GRAD_X, None, -3)):
        desc = _lib.EnfDesc(**{**OK, "flags": flags})
        rc = lib.enf_xattn_bwd_x(ctypes.byref(desc), ctypes.byref(w), 16, 0, 16, 16, 16, 16, None, 16, 16, 16, dx, 256, 1 << 40, None)
        assert rc == want, lib.enf_last_error()


def oracle_grad_x(cfg, params, x, p, a, sigma, d_out):
    """d<d_out, nef_apply>/dx by torch autograd through the oracle (invariant() and gaussian_window() see x)."""
    xg = x.detach().clone().requires_grad_(True)
    out = R.nef_apply(cfg, params, xg, p, a, sigma)
    (dx,) = torch.autograd.grad(out, xg, grad_outputs=d_out)
    return dx


@pytest.mark.parametrize("name", golden_names() + golden_names(sa=True))
def test_oracle_grad_x_matches_finite_differences(name):
    """The oracle's x-gradient against fp64 central differences of the oracle forward, whose output the golden fixtures pin
    to the reference's own module code.  Small cases: the first 6 queries of every field."""
    cfg, params, _, rec = load_golden(name)
    x, p, a, sigma, cot = rec["x"][:, :6], rec["p"], rec["a"], rec["sigma"], rec["cot"][:, :6]
    dx = oracle_grad_x(cfg, params, x, p, a, sigma, cot)
    loss = lambda xx: float((R.nef_apply(cfg, params, xx, p, a, sigma) * cot).sum())
    h = 1e-6
    fd = torch.zeros_like(x)
    for idx in torch.cartesian_prod(*(torch.arange(n) for n in x.shape)).tolist():
        xp, xm = x.clone(), x.clone()
        xp[tuple(idx)] += h
        xm[tuple(idx)] -= h
        fd[tuple(idx)] = (loss(xp) - loss(xm)) / (2 * h)
    assert float(dx.abs().max()) > 0
    assert rel_err(dx, fd) < 2e-6, rel_err(dx, fd)
