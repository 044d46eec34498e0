"""Drop-in host API for the ENF cross-attention path: the reference's `init` / `apply` surface over
the hand-written CUDA kernels (C ABI in include/enf_b200.h).

Mirrors `EquivariantCrossAttentionNeF` (enf/models/equivariant_cross_attention_nef.py:70-235):
same constructor fields, same argument order `(x, p, a, gaussian_window_size)`, same parameter
tree (`{'params': {...}}` with Flax's names, SURVEY.md A.3) and the same latent layout
`p (B,Z,P_raw)`, `a (B,Z,L)`, `gaussian_window (B,Z,1)` (enf/latents/autodecoder.py:58-73).
PyTorch is used only as plumbing (device memory, streams, autograd tape); all arithmetic of the path
runs in libenf_b200.so.  The op is ONCE differentiable: first-order gradients w.r.t. parameters,
p, a, the window size and the coordinates x (spatial derivatives of the decoded field; computed only
when x requires grad, ENF_FLAG_GRAD_X).  For a shared 2-D grid x the gradient is the sum over fields.
"""
import ctypes
import math
import weakref
from typing import Dict, Optional, Sequence

import torch

from . import _lib
from .invariant import BaseInvariant


def _flatten(tree, prefix=""):
    out = {}
    for k, v in tree.items():
        name = f"{prefix}/{k}" if prefix else k
        if isinstance(v, dict):
            out.update(_flatten(v, name))
        else:
            out[name] = v
    return out


def _unflatten(flat):
    out = {}
    for name, v in flat.items():
        node = out
        parts = name.split("/")
        for k in parts[:-1]:
            node = node.setdefault(k, {})
        node[parts[-1]] = v
    return out


def params_to_leaves(variables, paths=None) -> list:
    """Flax-style tree -> the 46 leaves in EnfWeights order (None for leaves the call does not use, see _lib.leaf_paths)."""
    flat = _flatten(variables["params"] if "params" in variables else variables)
    paths = _lib.LEAF_PATHS if paths is None else paths
    try:
        return [None if paths[n] is None else flat[paths[n]] for n in _lib.LEAVES]
    except KeyError as e:
        raise KeyError(f"parameter tree is missing {e}; expected the tree produced by nef.init") from None


def leaves_to_params(leaves: Sequence) -> Dict:
    return {"params": _unflatten({_lib.LEAF_PATHS[n]: t for n, t in zip(_lib.LEAVES, leaves)})}


def _ptr(t: Optional[torch.Tensor]):
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def _weights_struct(leaves):
    w = _lib.EnfWeights()
    for n, t in zip(_lib.LEAVES, leaves):
        setattr(w, n, 0 if t is None else t.data_ptr())
    return w


def _as_f32(t, name):
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: the ENF path has no CPU implementation in this package")
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32 (the reference computes in float32), got {t.dtype}")
    return t.contiguous()


class _XAttnFunction(torch.autograd.Function):
    """enf_xattn_fwd / enf_xattn_bwd (enf_xattn_bwd_x when x needs a gradient) on torch's current stream."""

    @staticmethod
    def forward(ctx, meta, x, p, a, sigma, *leaves):
        lib = _lib.load()
        desc_kw, x_shared = meta
        desc = _lib.EnfDesc(**desc_kw)
        ctx.n_extra = 0
        if desc.flags & _lib.FLAG_FROZEN_RELU:          # trailing argument: the mask poses; the C ABI takes p[2][B,Z,P]
            *leaves, p_mask = leaves
            ctx.n_extra = 1
            ctx.p_shape = tuple(p.shape)
            p = torch.stack([_as_f32(p, "p"), _as_f32(p_mask, "relu_mask_pose")]).contiguous()
        p = _as_f32(p, "p"); a = _as_f32(a, "a")
        x = p if x is None else _as_f32(x, "x")          # latent self-attention step: the queries are the poses
        sigma = None if sigma is None else _as_f32(sigma, "gaussian_window_size")
        ctx.leaf_mask = [t is not None for t in leaves]
        leaves = [None if t is None else _as_f32(t, n) for t, n in zip(leaves, _lib.LEAVES)]
        nbytes = lib.enf_xattn_workspace_bytes(ctypes.byref(desc))
        if nbytes == 0:
            raise _lib.EnfLibraryError("bad problem description: " + lib.enf_last_error().decode())
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        # the library keys its forward state on the workspace address: drop the entry when the buffer dies, so that a later
        # allocation at the same address can never pass for this forward
        weakref.finalize(ws, lib.enf_workspace_release, ctypes.c_void_p(ws.data_ptr()))
        out_dtype = torch.bfloat16 if desc.flags & _lib.FLAG_OUT_BF16 else torch.float32
        out = torch.empty(desc.B, desc.C, desc.O, dtype=out_dtype, device=p.device)
        w = _weights_struct(leaves)
        stream = ctypes.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)
        xbs = 0 if x_shared else desc.C * desc.Dx
        with torch.cuda.device(x.device):
            rc = lib.enf_xattn_fwd(ctypes.byref(desc), ctypes.byref(w), _ptr(x), xbs, _ptr(p), _ptr(a), _ptr(sigma),
                                   _ptr(out), _ptr(ws), nbytes, stream)
        _lib.check(rc, "enf_xattn_fwd")
        ctx.desc_kw, ctx.xbs, ctx.ws, ctx.nbytes = desc_kw, xbs, ws, nbytes
        ctx.has_sigma = sigma is not None
        ctx.save_for_backward(x, p, a, *([sigma] if sigma is not None else []), *[t for t in leaves if t is not None])
        ctx.launches_fwd = lib.enf_last_launch_count()
        _XAttnFunction.last_launches = [ctx.launches_fwd, 0]
        ctx.forward_only = bool(desc_kw.get("flags", 0) & _lib.FLAG_FORWARD_ONLY)
        # diagnostics (enf_debug_ws_offset views, tests): a WEAK reference -- the workspace (GBs) dies with its autograd node
        _XAttnFunction.last_ws = (desc_kw, weakref.ref(ws), nbytes)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, d_out):
        # repeatable (retain_graph=True): enf_xattn_bwd leaves the forward state in the workspace intact
        lib = _lib.load()
        saved = list(ctx.saved_tensors)
        x, p, a = saved[:3]
        sigma = saved[3] if ctx.has_sigma else None
        it = iter(saved[4:] if ctx.has_sigma else saved[3:])
        leaves = [next(it) if used else None for used in ctx.leaf_mask]
        desc = _lib.EnfDesc(**ctx.desc_kw)
        d_out = _as_f32(d_out, "d_out")
        need_w = any(ctx.needs_input_grad[5:5 + len(leaves)])
        grads = [None if t is None else torch.empty_like(t) for t in leaves] if need_w else None
        dp = torch.empty(ctx.p_shape, dtype=p.dtype, device=p.device) if ctx.n_extra else torch.empty_like(p)
        da = torch.empty_like(a)
        dsigma = torch.empty_like(sigma) if sigma is not None else None
        # x: [B,C,Dx], or the shared grid [C,Dx] (then dx sums the fields; the caller's expand carries it back)
        dx = torch.empty_like(x) if ctx.needs_input_grad[1] and desc.flags & _lib.FLAG_GRAD_X else None
        w = _weights_struct(leaves)
        gw = _weights_struct(grads) if need_w else None
        stream = ctypes.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)
        with torch.cuda.device(x.device):
            args = (ctypes.byref(desc), ctypes.byref(w), _ptr(x), ctx.xbs, _ptr(p), _ptr(a), _ptr(sigma), _ptr(d_out),
                    ctypes.byref(gw) if need_w else None, _ptr(dp), _ptr(da), _ptr(dsigma))
            if dx is not None:
                rc = lib.enf_xattn_bwd_x(*args, _ptr(dx), _ptr(ctx.ws), ctx.nbytes, stream)
            else:
                rc = lib.enf_xattn_bwd(*args, _ptr(ctx.ws), ctx.nbytes, stream)
        _lib.check(rc, "enf_xattn_bwd_x" if dx is not None else "enf_xattn_bwd")
        _XAttnFunction.last_launches[1] = lib.enf_last_launch_count()
        return (None, dx, dp, da, dsigma, *(grads if need_w else [None] * len(leaves)), *([None] * ctx.n_extra))


_XAttnFunction.last_launches = [0, 0]


def last_launch_counts():
    """(kernels enqueued by the last forward, by the last backward) -- for bench.py's gpu_launches."""
    return tuple(_XAttnFunction.last_launches)


class EquivariantCrossAttentionNeF:
    """Same constructor fields as the reference module (equivariant_cross_attention_nef.py:85-96)."""

    def __init__(self, num_hidden: int, num_heads: int, num_layers: int, num_out: int, latent_dim: int,
                 cross_attn_invariant: BaseInvariant, self_attn_invariant: Optional[BaseInvariant] = None,
                 embedding_type: str = "rff", embedding_freq_multiplier=(0.05, 0.1),
                 condition_value_transform: bool = True, use_gaussian_window: bool = True,
                 precision: str = "fp32", recompute: bool = False, chunk_fields: int = 0,
                 workspace_cap_bytes: Optional[int] = None, out_bf16: bool = False, forward_chunk_fields: int = 0):
        if num_layers < 0:
            raise ValueError("num_layers must be >= 0")
        if num_layers > 0 and self_attn_invariant is None:
            raise ValueError("num_layers > 0 needs the self-attention invariant (get_sa_invariant)")
        if embedding_type != "rff":
            raise ValueError(f"Unknown embedding type: {embedding_type}." if embedding_type not in ("ffn", "polynomial")
                             else f"embedding_type '{embedding_type}' is not on the accelerated path (configs use 'rff')")
        if not condition_value_transform:
            raise NotImplementedError("condition_value_transform=False is not on the accelerated path")
        if num_hidden % 2:
            raise AssertionError("For the Fourier Features hidden_dim should be even to calculate them correctly.")
        self.num_hidden, self.num_heads, self.num_layers = num_hidden, num_heads, num_layers
        self.num_out, self.latent_dim = num_out, latent_dim
        self.cross_attn_invariant, self.self_attn_invariant = cross_attn_invariant, self_attn_invariant
        self.embedding_type = embedding_type
        self.embedding_freq_multiplier = tuple(embedding_freq_multiplier)
        self.condition_value_transform = condition_value_transform
        self.use_gaussian_window = use_gaussian_window
        self.precision = {"fp32": _lib.PREC_FP32, "bf16": _lib.PREC_BF16}[precision]
        # bounded-memory training (ENF_FLAG_RECOMPUTE): no per-(query, latent) stash; the backward re-runs the pair forward
        # per chunk of `chunk_fields` fields (0: library default), or of as many fields as fit `workspace_cap_bytes`
        self.recompute = bool(recompute) or workspace_cap_bytes is not None
        self.chunk_fields, self.workspace_cap_bytes = int(chunk_fields), workspace_cap_bytes
        self.out_bf16 = bool(out_bf16)       # forward-only calls return bfloat16 (ENF_FLAG_OUT_BF16, num_out <= 4)
        # forward-only calls (validation roll-outs decode B*T fields at once, _base_pde_trainer.py:446-457) walk the fields in
        # chunks of this many, so the workspace is that of one chunk whatever B*T is (0: one call)
        self.forward_chunk_fields = int(forward_chunk_fields)

    # -- nef.init(key, x, p, a, window) (pde_trainer.py:99-102) -----------------------------------------
    def init(self, key, x, p, a, gaussian_window_size=None):
        """Parameter tree with Flax's names, shapes and initialisers.  `key`: int seed or torch.Generator."""
        dev = a.device
        g = key if isinstance(key, torch.Generator) else torch.Generator().manual_seed(int(key))
        d, H, L, O = self.num_hidden, self.num_heads, self.latent_dim, self.num_out
        I = self.cross_attn_invariant.dim
        if a.shape[-1] != L:
            raise ValueError(f"a has latent_dim {a.shape[-1]}, module was built with {L}")

        fq, fv = self.embedding_freq_multiplier

        def normal(shape, std):
            return torch.randn(shape, generator=g) * std

        def lecun(n_in, n_out):      # flax default kernel_init: variance_scaling(1, fan_in, truncated_normal)
            t = torch.empty(n_in, n_out)
            torch.nn.init.trunc_normal_(t, mean=0.0, std=1.0, a=-2.0, b=2.0, generator=g)
            return t * (math.sqrt(1.0 / n_in) / 0.87962566103423978)

        def dense(n_in, n_out):
            return {"kernel": lecun(n_in, n_out), "bias": torch.zeros(n_out)}

        def ffn(n_in, n_hid, n_out):
            return {"Dense_0": dense(n_in, n_hid), "LayerNorm_0": {"scale": torch.ones(n_hid), "bias": torch.zeros(n_hid)},
                    "Dense_1": dense(n_hid, n_out)}

        def rff(std, I=I):           # rff.py:35-40,55-60,83
            return {"encoding": {"coefficients": normal((I, d // 2), std)},
                    "layers_0": {"linear": {"kernel": normal((d, d), math.sqrt(2.0 / d)), "bias": normal((d,), 1e-6)}},
                    "linear_final": {"kernel": (torch.rand(d, d, generator=g) * 2 - 1) * math.sqrt(6.0 / d),
                                     "bias": normal((d,), 1e-6)}}

        fq, fv = self.embedding_freq_multiplier
        def self_block():            # residual=True, project_heads=True (equivariant_cross_attention_nef.py:159-167, 35-37, 68-70)
            Is = 3 if self.self_attn_invariant.invariant_type == "ponita" else self.self_attn_invariant.dim
            return {"layer_norm_attn": {"scale": torch.ones(d), "bias": torch.zeros(d)},
                    "attn": {"invariant_embedding_query": rff(fq, Is), "invariant_embedding_value": rff(fv, Is),
                             "inv_emb_to_q": dense(d, H * d), "a_to_k": dense(d, H * d), "a_to_v": dense(d, H * d),
                             "inv_emb_to_v": ffn(d, d, 2 * H * d), "inv_emb_cond_mixer": ffn(d, d, d),
                             "out_proj": dense(H * d, d)},
                    "pointwise_ffn": ffn(d, d, d)}

        tree = {
            "latent_stem": dense(L, d),
            **{f"self_attention_blocks_{i}": self_block() for i in range(self.num_layers)},
            "cross_attention_blocks_0": {
                "layer_norm_attn": {"scale": torch.ones(d), "bias": torch.zeros(d)},
                "attn": {
                    "invariant_embedding_query": rff(fq), "invariant_embedding_value": rff(fv),
                    "inv_emb_to_q": dense(d, H * d), "a_to_k": dense(d, H * d), "a_to_v": dense(d, H * d),
                    "inv_emb_to_v": ffn(d, d, 2 * H * d), "inv_emb_cond_mixer": ffn(d, d, d),
                    "out_proj": dense(H * d, H * d)},
                "pointwise_ffn": ffn(H * d, H * d, H * d)},
            "out_proj": {"layers_0": dense(H * d, d), "layers_2": dense(d, d), "layers_4": dense(d, O)},
        }
        flat = {k: v.to(device=dev, dtype=torch.float32).contiguous() for k, v in _flatten(tree).items()}
        return {"params": _unflatten(flat)}

    # -- nef.apply(params, x, p, a, window) (pde_trainer.py:184,478,537) -----------------------------------
    def apply(self, variables, x, p, a, gaussian_window_size=None, relu_mask_pose=None):
        """`relu_mask_pose` (B,Z,P), fp32 precision only: evaluate with the relu activation pattern of THOSE poses
        (ENF_FLAG_FROZEN_RELU; used by enf_pde_b200.meta for Hessian-vector products)."""
        inv = self.cross_attn_invariant
        if self.use_gaussian_window and gaussian_window_size is None:
            raise TypeError("gaussian_window_size is None but use_gaussian_window=True "
                            "(the reference fails on `sigma[:, None, :]` in the same situation)")
        if x.dim() == 2:
            x = x.unsqueeze(0).expand(p.shape[0], *x.shape)
        B, C, Dx = x.shape
        if p.shape[0] != B or a.shape[0] != B:
            raise ValueError("x, p, a must share the leading (field) dimension")
        Z = p.shape[1]
        if p.shape[2] != inv.pose_dim:
            raise ValueError(f"p has pose width {p.shape[2]}, invariant '{inv.invariant_type}' expects {inv.pose_dim}")
        x_shared = x.stride(0) == 0 and B > 1
        x_arg = x[0] if x_shared else x
        sigma = gaussian_window_size if self.use_gaussian_window else None
        if sigma is not None and tuple(sigma.shape) != (B, Z, 1):
            raise ValueError(f"gaussian_window_size must have shape {(B, Z, 1)}")
        # gradient w.r.t. the coordinates: set at forward time (the workspace then holds the query-record cotangents)
        grad_x = torch.is_grad_enabled() and x.requires_grad
        desc = dict(B=B, C=C, Z=Z, d=self.num_hidden, H=self.num_heads, L=self.latent_dim, O=self.num_out, Dx=Dx,
                    invariant_kind=_lib.INVARIANT_KINDS[inv.invariant_type], use_window=int(self.use_gaussian_window),
                    precision=self.precision, flags=_lib.FLAG_GRAD_X if grad_x else 0)
        if self.num_layers > 0:
            # latent self-attention steps first (equivariant_cross_attention_nef.py:223-226): a <- gelu(a + block_i(p, p, a)); each is one
            # call of the same C entry points with ENF_FLAG_SELF_BLOCK; the first applies latent_stem, the decode call below none
            if relu_mask_pose is not None or self.recompute:
                raise NotImplementedError("relu_mask_pose / recompute are not combined with num_layers > 0")
            if self.self_attn_invariant.invariant_type != inv.invariant_type:
                raise ValueError("self- and cross-attention invariants must come from the same cfg.nef.invariant_type")
            grad_on = torch.is_grad_enabled()
            for i in range(self.num_layers):
                sdesc = dict(desc, C=Z, O=self.num_hidden, L=(self.latent_dim if i == 0 else self.num_hidden),
                             flags=_lib.FLAG_SELF_BLOCK | (0 if i == 0 else _lib.FLAG_NO_STEM))
                sl = params_to_leaves(variables, _lib.leaf_paths(f"self_attention_blocks_{i}", with_stem=(i == 0), with_mlp=False))
                if not (grad_on and any(t is not None and t.requires_grad for t in (p, a, sigma, *sl))):
                    sdesc["flags"] |= _lib.FLAG_FORWARD_ONLY
                a = _XAttnFunction.apply((sdesc, False), None, p, a, sigma, *sl)
            desc["L"] = self.num_hidden
            desc["flags"] |= _lib.FLAG_NO_STEM
            leaves = params_to_leaves(variables, _lib.leaf_paths("cross_attention_blocks_0", with_stem=False, with_mlp=True))
        else:
            leaves = params_to_leaves(variables)
        if relu_mask_pose is not None:
            if tuple(relu_mask_pose.shape) != tuple(p.shape):
                raise ValueError("relu_mask_pose must have the shape of p")
            desc["flags"] |= _lib.FLAG_FROZEN_RELU
            return _XAttnFunction.apply((desc, x_shared), x_arg, p, a, sigma, *leaves, relu_mask_pose.detach())
        # forward only (validation roll-outs, pde_trainer.py:389-405): nothing is kept for a backward
        if not (grad_x or torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in (p, a, sigma, *leaves))):
            desc["flags"] |= _lib.FLAG_FORWARD_ONLY
            if self.out_bf16:
                desc["flags"] |= _lib.FLAG_OUT_BF16
            n = self.forward_chunk_fields
            if 0 < n < B and self.num_layers == 0:
                outs = []
                for b0 in range(0, B, n):
                    sl = slice(b0, min(B, b0 + n))
                    cd = dict(desc, B=sl.stop - sl.start)
                    outs.append(_XAttnFunction.apply((cd, x_shared), x_arg if x_shared else x_arg[sl], p[sl], a[sl],
                                                     None if sigma is None else sigma[sl], *leaves))
                return torch.cat(outs, dim=0)
        elif self.recompute:
            desc["flags"] |= _lib.FLAG_RECOMPUTE
            desc["chunk_fields"] = self.chunk_fields
            if self.workspace_cap_bytes is not None:
                n = _lib.load().enf_xattn_chunk_for_cap(ctypes.byref(_lib.EnfDesc(**desc)), int(self.workspace_cap_bytes))
                if n <= 0:
                    raise _lib.EnfLibraryError(f"workspace_cap_bytes={self.workspace_cap_bytes} is too small for this problem "
                                               "even with one field per backward chunk")
                desc["chunk_fields"] = n
        return _XAttnFunction.apply((desc, x_shared), x_arg, p, a, sigma, *leaves)

    __call__ = apply
