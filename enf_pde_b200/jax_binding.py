"""jax.ffi binding of the B200 ENF path: what the reference's JAX host code imports instead of calling the Flax module.

    from enf_pde_b200.jax_binding import make_enf_apply
    enf_apply = make_enf_apply(nef_cfg, invariant_type, num_in)          # once
    out = enf_apply(leaves, x, p, a, sigma)                               # replaces self.nef.apply(...) in loss_fn,
                                                                          # experiments/fitting/trainers/pde_trainer.py:184

`leaves` = the 46 arrays of `nef.init(...)['params']` in EnfWeights order (`enf_pde_b200._lib.LEAF_PATHS` maps each to its
Flax path).  The op is once-differentiable (`jax.custom_vjp`): gradients w.r.t. leaves, p, a, sigma -- what `jax.grad` at
pde_trainer.py:188,255 takes.  Known gap: the cotangent of the coordinates x is returned as zeros here.  The C ABI has it
(ENF_FLAG_GRAD_X + enf_xattn_bwd_x, which the PyTorch binding uses), but the FFI handler of csrc/enf_xla_ffi.cc does not yet
request it; differentiate x through enf_pde_b200.nef until it does.

This module needs JAX and the shim library built from csrc/enf_xla_ffi.cc (see its header).  Neither exists in the image
this repo was developed in (no jax wheel, no network), so this file is exercised only where JAX is installed; everything
the repo tests goes through the same C ABI from PyTorch (enf_pde_b200/nef.py).
"""
import ctypes
import os

from . import _lib

try:                                      # pragma: no cover - JAX is not installable in the development image
    import jax
    import jax.numpy as jnp
    import numpy as np
    HAVE_JAX = True
except ImportError:                       # pragma: no cover
    HAVE_JAX = False

_SHIM = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libenf_b200_xla.so")
_registered = False


def _register():
    global _registered
    if _registered:
        return
    if not HAVE_JAX:
        raise ImportError("enf_pde_b200.jax_binding needs jax (jax.ffi); the PyTorch binding is enf_pde_b200.nef")
    if not os.path.exists(_SHIM):
        raise FileNotFoundError(f"{_SHIM} not built: see the build line at the top of csrc/enf_xla_ffi.cc")
    _lib.load()                            # libenf_b200.so first: the shim links against it
    shim = ctypes.CDLL(_SHIM)
    jax.ffi.register_ffi_target("enf_xattn_fwd", jax.ffi.pycapsule(shim.EnfXattnFwd), platform="CUDA")
    jax.ffi.register_ffi_target("enf_xattn_bwd", jax.ffi.pycapsule(shim.EnfXattnBwd), platform="CUDA")
    jax.ffi.register_ffi_target("enf_ode_fwd", jax.ffi.pycapsule(shim.EnfOdeFwd), platform="CUDA")
    jax.ffi.register_ffi_target("enf_ode_bwd", jax.ffi.pycapsule(shim.EnfOdeBwd), platform="CUDA")
    _registered = True


def make_enf_apply(num_hidden, num_heads, num_out, latent_dim, invariant_type, num_in, use_gaussian_window=True,
                   precision="bf16", recompute=False, chunk_fields=0):
    """Returns enf_apply(leaves, x, p, a, sigma) -> (B, C, num_out), differentiable once in leaves, p, a, sigma.
    recompute: ENF_FLAG_RECOMPUTE (the workspace -- a custom_vjp residual, several of which are live inside inner_loop -- then
    scales with chunk_fields fields instead of the batch)."""
    _register()
    lib = _lib.load()
    kind = _lib.INVARIANT_KINDS[invariant_type]
    prec = {"fp32": _lib.PREC_FP32, "bf16": _lib.PREC_BF16}[precision]
    flags = _lib.FLAG_RECOMPUTE if recompute else 0
    attrs = dict(d=np.int32(num_hidden), H=np.int32(num_heads), L=np.int32(latent_dim), O=np.int32(num_out),
                 invariant_kind=np.int32(kind), use_window=np.int32(int(use_gaussian_window)), precision=np.int32(prec),
                 flags=np.int32(flags), chunk_fields=np.int32(chunk_fields))

    def ws_bytes(B, C, Z):
        desc = _lib.EnfDesc(B=B, C=C, Z=Z, d=num_hidden, H=num_heads, L=latent_dim, O=num_out, Dx=num_in, invariant_kind=kind,
                            use_window=int(use_gaussian_window), precision=prec, flags=flags, chunk_fields=chunk_fields)
        n = lib.enf_xattn_workspace_bytes(ctypes.byref(desc))
        if n == 0:
            raise ValueError(lib.enf_last_error().decode())
        return n

    def fwd_call(leaves, x, p, a, sigma):
        B, Z = p.shape[0], p.shape[1]
        C = x.shape[-2]
        sig = sigma if use_gaussian_window else jnp.zeros((0,), jnp.float32)
        return jax.ffi.ffi_call(
            "enf_xattn_fwd",
            (jax.ShapeDtypeStruct((B, C, num_out), jnp.float32), jax.ShapeDtypeStruct((ws_bytes(B, C, Z),), jnp.uint8)),
        )(x, p, a, sig, *leaves, **attrs)

    @jax.custom_vjp
    def enf_apply(leaves, x, p, a, sigma):
        return fwd_call(leaves, x, p, a, sigma)[0]

    def vjp_fwd(leaves, x, p, a, sigma):
        out, ws = fwd_call(leaves, x, p, a, sigma)
        return out, (ws, leaves, x, p, a, sigma)

    def vjp_bwd(res, d_out):
        ws, leaves, x, p, a, sigma = res
        sig = sigma if use_gaussian_window else jnp.zeros((0,), jnp.float32)
        # result 0 = the workspace again, aliased to operand 4: the backward's scratch writes then go to a buffer XLA knows
        # is written (an input operand may be aliased / CSE'd); XLA copies the donated residual if it is still live
        shapes = [jax.ShapeDtypeStruct(ws.shape, jnp.uint8)]
        shapes += [jax.ShapeDtypeStruct(l.shape, jnp.float32) for l in leaves]
        shapes += [jax.ShapeDtypeStruct(p.shape, jnp.float32), jax.ShapeDtypeStruct(a.shape, jnp.float32),
                   jax.ShapeDtypeStruct(sig.shape, jnp.float32)]
        outs = jax.ffi.ffi_call("enf_xattn_bwd", tuple(shapes), input_output_aliases={4: 0})(x, p, a, sig, ws, d_out, *leaves, **attrs)
        outs = outs[1:]
        n = len(leaves)
        dsigma = outs[n + 2] if use_gaussian_window else None
        return (list(outs[:n]), jnp.zeros_like(x), outs[n], outs[n + 1], dsigma)     # x: see the module docstring

    enf_apply.defvjp(vjp_fwd, vjp_bwd)
    return enf_apply


def make_ode_apply(num_hidden, num_layers, latent_dim, invariant_type, num_in, basis_dim, degree, widening_factor):
    """Returns ode_apply(leaves, p, a) -> (dp/dt, da/dt), differentiable once in leaves, p, a: the body of
    `ode_model.apply(params, (p, a, window))` for PonitaODEGen (ponita_ode_g.py:229-257; the window's derivative is zeros_like(window),
    which the caller adds).  `leaves`: the arrays of `params['ponita']` in EnfOdeWeights order (`enf_pde_b200.ode.leaf_paths`).
    Reference-side use (pde_trainer.py:381,433,582):  f=lambda z, t: (*ode_apply(leaves, z[0], z[1]), jnp.zeros_like(z[2]))"""
    _register()
    from . import ode as _ode
    lib = _ode._load()
    kind = _lib.INVARIANT_KINDS[invariant_type]
    attrs = dict(hidden=np.int32(num_hidden), basis=np.int32(basis_dim), layers=np.int32(num_layers), widen=np.int32(widening_factor),
                 degree=np.int32(degree), Dx=np.int32(num_in), invariant_kind=np.int32(kind))

    def ws_bytes(B, Z):
        desc = _ode.EnfOdeDesc(B=B, Z=Z, L=latent_dim, hidden=num_hidden, basis=basis_dim, layers=num_layers, widen=widening_factor,
                               degree=degree, Dx=num_in, invariant_kind=kind)
        n = lib.enf_ode_workspace_bytes(ctypes.byref(desc))
        if n == 0:
            raise ValueError(lib.enf_last_error().decode())
        return n

    def fwd_call(leaves, p, a):
        shapes = (jax.ShapeDtypeStruct(p.shape, jnp.float32), jax.ShapeDtypeStruct(a.shape, jnp.float32),
                  jax.ShapeDtypeStruct((ws_bytes(p.shape[0], p.shape[1]),), jnp.uint8))
        return jax.ffi.ffi_call("enf_ode_fwd", shapes)(p, a, *leaves, **attrs)

    @jax.custom_vjp
    def ode_apply(leaves, p, a):
        return fwd_call(leaves, p, a)[:2]

    def vjp_fwd(leaves, p, a):
        dp, da, ws = fwd_call(leaves, p, a)
        return (dp, da), (ws, leaves, p, a)

    def vjp_bwd(res, cot):
        ws, leaves, p, a = res
        g_dp, g_da = cot
        shapes = [jax.ShapeDtypeStruct(ws.shape, jnp.uint8)] + [jax.ShapeDtypeStruct(l.shape, jnp.float32) for l in leaves]
        shapes += [jax.ShapeDtypeStruct(p.shape, jnp.float32), jax.ShapeDtypeStruct(a.shape, jnp.float32)]
        outs = jax.ffi.ffi_call("enf_ode_bwd", tuple(shapes), input_output_aliases={2: 0})(p, a, ws, g_dp, g_da, *leaves, **attrs)[1:]
        n = len(leaves)
        return (list(outs[:n]), outs[n], outs[n + 1])

    ode_apply.defvjp(vjp_fwd, vjp_bwd)
    return ode_apply
