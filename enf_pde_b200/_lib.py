"""ctypes binding of the C ABI in include/enf_b200.h (libenf_b200.so, built in-tree by `make -C csrc`).

There is deliberately no fallback: if the shared library is missing or a call fails, this raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libenf_b200.so")

# order == field order of EnfWeights / EnfWeightGrads in include/enf_b200.h
LEAVES = (
    "stem_w", "stem_b", "ln_attn_g", "ln_attn_b",
    "q_omega", "q_w1", "q_b1", "q_wf", "q_bf",
    "v_omega", "v_w1", "v_b1", "v_wf", "v_bf",
    "wq", "bq", "wk", "bk", "wv", "bv",
    "fv_w1", "fv_b1", "fv_g", "fv_beta", "fv_w2", "fv_b2",
    "mx_w1", "mx_b1", "mx_g", "mx_beta", "mx_w2", "mx_b2",
    "wo", "bo",
    "fb_w1", "fb_b1", "fb_g", "fb_beta", "fb_w2", "fb_b2",
    "m0_w", "m0_b", "m1_w", "m1_b", "m2_w", "m2_b",
)

# leaf -> path in the Flax parameter tree produced by nef.init (SURVEY.md A.3)
_A = "cross_attention_blocks_0/attn/"
LEAF_PATHS = {
    "stem_w": "latent_stem/kernel", "stem_b": "latent_stem/bias",
    "ln_attn_g": "cross_attention_blocks_0/layer_norm_attn/scale",
    "ln_attn_b": "cross_attention_blocks_0/layer_norm_attn/bias",
    "q_omega": _A + "invariant_embedding_query/encoding/coefficients",
    "q_w1": _A + "invariant_embedding_query/layers_0/linear/kernel",
    "q_b1": _A + "invariant_embedding_query/layers_0/linear/bias",
    "q_wf": _A + "invariant_embedding_query/linear_final/kernel",
    "q_bf": _A + "invariant_embedding_query/linear_final/bias",
    "v_omega": _A + "invariant_embedding_value/encoding/coefficients",
    "v_w1": _A + "invariant_embedding_value/layers_0/linear/kernel",
    "v_b1": _A + "invariant_embedding_value/layers_0/linear/bias",
    "v_wf": _A + "invariant_embedding_value/linear_final/kernel",
    "v_bf": _A + "invariant_embedding_value/linear_final/bias",
    "wq": _A + "inv_emb_to_q/kernel", "bq": _A + "inv_emb_to_q/bias",
    "wk": _A + "a_to_k/kernel", "bk": _A + "a_to_k/bias",
    "wv": _A + "a_to_v/kernel", "bv": _A + "a_to_v/bias",
    "fv_w1": _A + "inv_emb_to_v/Dense_0/kernel", "fv_b1": _A + "inv_emb_to_v/Dense_0/bias",
    "fv_g": _A + "inv_emb_to_v/LayerNorm_0/scale", "fv_beta": _A + "inv_emb_to_v/LayerNorm_0/bias",
    "fv_w2": _A + "inv_emb_to_v/Dense_1/kernel", "fv_b2": _A + "inv_emb_to_v/Dense_1/bias",
    "mx_w1": _A + "inv_emb_cond_mixer/Dense_0/kernel", "mx_b1": _A + "inv_emb_cond_mixer/Dense_0/bias",
    "mx_g": _A + "inv_emb_cond_mixer/LayerNorm_0/scale", "mx_beta": _A + "inv_emb_cond_mixer/LayerNorm_0/bias",
    "mx_w2": _A + "inv_emb_cond_mixer/Dense_1/kernel", "mx_b2": _A + "inv_emb_cond_mixer/Dense_1/bias",
    "wo": _A + "out_proj/kernel", "bo": _A + "out_proj/bias",
    "fb_w1": "cross_attention_blocks_0/pointwise_ffn/Dense_0/kernel",
    "fb_b1": "cross_attention_blocks_0/pointwise_ffn/Dense_0/bias",
    "fb_g": "cross_attention_blocks_0/pointwise_ffn/LayerNorm_0/scale",
    "fb_beta": "cross_attention_blocks_0/pointwise_ffn/LayerNorm_0/bias",
    "fb_w2": "cross_attention_blocks_0/pointwise_ffn/Dense_1/kernel",
    "fb_b2": "cross_attention_blocks_0/pointwise_ffn/Dense_1/bias",
    "m0_w": "out_proj/layers_0/kernel", "m0_b": "out_proj/layers_0/bias",
    "m1_w": "out_proj/layers_2/kernel", "m1_b": "out_proj/layers_2/bias",
    "m2_w": "out_proj/layers_4/kernel", "m2_b": "out_proj/layers_4/bias",
}

# leaves a latent self-attention step does not use (no decode MLP) / a call with ENF_FLAG_NO_STEM does not use
_MLP_LEAVES = ("m0_w", "m0_b", "m1_w", "m1_b", "m2_w", "m2_b")
_STEM_LEAVES = ("stem_w", "stem_b")


def leaf_paths(block: str, with_stem: bool, with_mlp: bool):
    """leaf -> path (or None: unused by the call) for the block named `block` ('cross_attention_blocks_0', 'self_attention_blocks_<i>')."""
    out = {}
    for n, path in LEAF_PATHS.items():
        if (n in _STEM_LEAVES and not with_stem) or (n in _MLP_LEAVES and not with_mlp):
            out[n] = None
        else:
            out[n] = path.replace("cross_attention_blocks_0", block)
    return out


INVARIANT_KINDS = {
    "rel_pos": 0, "norm_rel_pos": 1, "abs_pos": 2, "rel_pos_periodic": 3, "ponita": 4,
    "polar_periodic": 5, "latitude_periodic": 6, "ball": 7, "ball_lat": 8,
}
PREC_FP32, PREC_BF16 = 0, 1
FLAG_FORWARD_ONLY = 1
FLAG_RECOMPUTE = 4
FLAG_OUT_BF16 = 8
FLAG_FROZEN_RELU = 16
FLAG_SELF_BLOCK = 32
FLAG_NO_STEM = 64
FLAG_GRAD_X = 128
ABI_VERSION = 2

EXPORTS = ("enf_abi_version", "enf_invariant_dim", "enf_pose_dim", "enf_xattn_workspace_bytes", "enf_xattn_chunk_for_cap",
           "enf_xattn_dispatch", "enf_workspace_release", "enf_xattn_fwd", "enf_xattn_bwd", "enf_xattn_bwd_x", "enf_last_launch_count",
           "enf_last_error", "enf_debug_ws_offset", "enf_profile_enable", "enf_profile_collect", "enf_debug_tc_gemm",
           "enf_debug_gemm")


class EnfDesc(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in
                ("B", "C", "Z", "d", "H", "L", "O", "Dx", "invariant_kind", "use_window", "precision", "flags",
                 "chunk_fields")] + [("reserved", ctypes.c_int32 * 3)]


class EnfWeights(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in LEAVES]


class EnfLibraryError(RuntimeError):
    pass


_lib = None


def load():
    """dlopen the in-tree library (once).  Raises EnfLibraryError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise EnfLibraryError(
            f"{LIB_PATH} is missing: build it with `make -C enf_pde_b200/csrc` (or __graft_entry__.build()). "
            "There is no CPU or PyTorch fallback for this path.")
    lib = ctypes.CDLL(LIB_PATH)
    lib.enf_abi_version.restype = ctypes.c_int
    lib.enf_invariant_dim.restype = ctypes.c_int
    lib.enf_invariant_dim.argtypes = [ctypes.c_int, ctypes.c_int]
    lib.enf_pose_dim.restype = ctypes.c_int
    lib.enf_pose_dim.argtypes = [ctypes.c_int, ctypes.c_int]
    lib.enf_xattn_workspace_bytes.restype = ctypes.c_size_t
    lib.enf_xattn_workspace_bytes.argtypes = [ctypes.POINTER(EnfDesc)]
    vp, i64 = ctypes.c_void_p, ctypes.c_int64
    lib.enf_xattn_chunk_for_cap.restype = ctypes.c_int
    lib.enf_xattn_chunk_for_cap.argtypes = [ctypes.POINTER(EnfDesc), ctypes.c_size_t]
    lib.enf_xattn_dispatch.restype = ctypes.c_int
    lib.enf_xattn_dispatch.argtypes = [ctypes.POINTER(EnfDesc), ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]
    lib.enf_workspace_release.restype = None
    lib.enf_workspace_release.argtypes = [vp]
    lib.enf_xattn_fwd.restype = ctypes.c_int
    lib.enf_xattn_fwd.argtypes = [ctypes.POINTER(EnfDesc), ctypes.POINTER(EnfWeights), vp, i64, vp, vp, vp, vp, vp,
                                  ctypes.c_size_t, vp]
    lib.enf_xattn_bwd.restype = ctypes.c_int
    lib.enf_xattn_bwd.argtypes = [ctypes.POINTER(EnfDesc), ctypes.POINTER(EnfWeights), vp, i64, vp, vp, vp, vp,
                                  ctypes.POINTER(EnfWeights), vp, vp, vp, vp, ctypes.c_size_t, vp]
    lib.enf_xattn_bwd_x.restype = ctypes.c_int
    lib.enf_xattn_bwd_x.argtypes = [ctypes.POINTER(EnfDesc), ctypes.POINTER(EnfWeights), vp, i64, vp, vp, vp, vp,
                                    ctypes.POINTER(EnfWeights), vp, vp, vp, vp, vp, ctypes.c_size_t, vp]
    lib.enf_last_launch_count.restype = ctypes.c_int
    lib.enf_last_error.restype = ctypes.c_char_p
    lib.enf_debug_ws_offset.restype = ctypes.c_int64
    lib.enf_debug_ws_offset.argtypes = [ctypes.POINTER(EnfDesc), ctypes.c_char_p, ctypes.POINTER(ctypes.c_int64)]
    lib.enf_profile_enable.restype = ctypes.c_int
    lib.enf_profile_enable.argtypes = [ctypes.c_int]
    lib.enf_profile_collect.restype = ctypes.c_int
    lib.enf_profile_collect.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_float), ctypes.c_int]
    lib.enf_debug_tc_gemm.restype = ctypes.c_int
    lib.enf_debug_tc_gemm.argtypes = [ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, vp]
    lib.enf_debug_gemm.restype = ctypes.c_int
    lib.enf_debug_gemm.argtypes = [ctypes.c_int] * 4 + [vp, i64, i64, vp, i64, i64, vp, vp, i64, vp, vp, vp, ctypes.c_int, vp]
    if lib.enf_abi_version() != ABI_VERSION:
        raise EnfLibraryError("libenf_b200.so ABI version mismatch")
    _lib = lib
    return lib


def dispatch(desc):
    """(pair forward on tcgen05?, pair backward on tcgen05?) for an EnfDesc -- what the library will actually run."""
    f, b = ctypes.c_int(0), ctypes.c_int(0)
    check(load().enf_xattn_dispatch(ctypes.byref(desc), ctypes.byref(f), ctypes.byref(b)), "enf_xattn_dispatch")
    return bool(f.value), bool(b.value)


def check(rc, what):
    if rc != 0:
        raise EnfLibraryError(f"{what} failed ({rc}): {load().enf_last_error().decode()}")
