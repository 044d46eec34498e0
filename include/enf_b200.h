/*
 * enf_b200.h -- C ABI of the B200-native ENF steerable cross-attention path.
 *
 * This is the drop-in boundary for the hot path of david-knigge/enf-pde:
 *   EquivariantCrossAttentionNeF.__call__      enf/models/equivariant_cross_attention_nef.py:204-235
 *     EquivariantCrossAttentionBlock.__call__  enf/models/equivariant_cross_attention_nef.py:44-67
 *       EquivariantCrossAttention.__call__     enf/steerable_attention/equivariant_cross_attention.py:74-151
 *         invariants + gaussian windows        enf/steerable_attention/invariant/ (all files)
 *         RFFNet                               enf/steerable_attention/embedding/rff.py:6-93
 * and of its reverse-mode derivative (jax.grad at experiments/fitting/trainers/pde_trainer.py:188,255).
 *
 * The reference has no FFI of its own (it is pure JAX); these entry points are what a
 * `jax.ffi` custom call (enf_pde_b200/csrc/enf_xla_ffi.cc) or any other host binding (ctypes in
 * enf_pde_b200/_lib.py) binds.  Conventions:
 *   - plain pointers and sizes only; every pointer except EnfDesc/EnfWeights/EnfWeightGrads
 *     themselves is DEVICE memory owned by the caller; the library never allocates, frees or
 *     retains device memory; scratch comes from the caller-provided workspace.
 *   - all tensors are dense row-major float32 with the reference's shapes.
 *   - functions only ENQUEUE work on `stream` (no device synchronisation, no default stream);
 *     they are re-entrant for distinct (workspace, stream) pairs.
 *   - return 0 on success, a negative ENF_ERR_* otherwise; no exceptions / exit() cross the ABI;
 *     enf_last_error() gives a thread-local message.  Asynchronous CUDA faults surface at the
 *     caller's next synchronisation.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef ENF_B200_H_
#define ENF_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ENF_B200_ABI_VERSION 2

/* cfg.nef.invariant_type -> get_ca_invariant (enf/steerable_attention/invariant/__init__.py:47-78) */
enum EnfInvariantKind {
  ENF_INV_REL_POS = 0,           /* RelativePositionND            rel_pos.py:26-41            */
  ENF_INV_NORM_REL_POS = 1,      /* NormRelativePositionND        norm_rel_pos.py:24-34       */
  ENF_INV_ABS_POS = 2,           /* AbsolutePositionND            abs_pos.py:27-42            */
  ENF_INV_REL_POS_PERIODIC = 3,  /* RelativePosition2DPeriodic    rel_pos_periodic.py:35-60   */
  ENF_INV_PONITA = 4,            /* PonitaPos2D                   ponita.py:20-44             */
  ENF_INV_POLAR_PERIODIC = 5,    /* RelativePositionPolarPeriodic polar_periodic.py:35-68     */
  ENF_INV_LATITUDE_PERIODIC = 6, /* RelativeLatitudePeriodic      spherical_longitude.py:34-85*/
  ENF_INV_BALL = 7,              /* BallInvariant                 ball.py:36-96               */
  ENF_INV_BALL_LAT = 8           /* BallLatInvariant              ball_lat.py:36-88           */
};

enum EnfPrecision {
  ENF_PREC_FP32 = 0,   /* fp32 FMA everywhere: the <= 1e-4 parity bucket                       */
  ENF_PREC_BF16 = 1    /* tcgen05 tensor cores, 16-bit operands, fp32 accumulate: <= 2e-3 bucket.  Pair kernels on the tensor
                          cores for num_hidden 32, 64, 128 and every num_heads 1..4 (beyond two heads at 64 / 128, and
                          four at 32, the forward and backward kernel A run once per group of <= 2 heads); num_hidden 16
                          runs the fp32 pair kernels.  enf_xattn_dispatch reports which. */
};

/* EnfDesc.flags */
enum EnfFlags {
  /* forward only: validation / visualisation roll-outs (apply_nef_jitted, pde_trainer.py:389-405;
   * _base_pde_trainer.py:446-457,588-598).  Nothing is saved for a backward (no logits, no operand
   * stash), the workspace is ~10x smaller, enf_xattn_bwd on such a workspace returns ENF_ERR_STATE. */
  ENF_FLAG_FORWARD_ONLY = 1,
  /* (bit 2 was ENF_FLAG_TC_BACKWARD_D64 in ABI 1: the tcgen05 backward is now the default at num_hidden = 64 too) */
  /* bounded-memory training (tensor-core precision mode): the forward keeps NO per-(query, latent) tensor for the
   * backward; enf_xattn_bwd walks the fields in chunks of EnfDesc.chunk_fields and re-runs the fused pair forward on each
   * chunk to rebuild that chunk's operand stash before its backward kernels.  The workspace then scales with
   * chunk_fields instead of B for everything that is O(B*C*Z) (use enf_xattn_chunk_for_cap to size it against a byte
   * budget); the price is one extra pair-forward pass per backward.  Results are bit-identical to the default (stash)
   * mode.  A no-op for the fp32 kernels, which always recompute. */
  ENF_FLAG_RECOMPUTE = 4,
  /* forward only, num_out <= 4: `out` is written as bfloat16 [B,C,O] instead of float32 (validation / visualisation
   * roll-outs decode B*T fields over the full grid, _base_pde_trainer.py:446-457). */
  ENF_FLAG_OUT_BF16 = 8,
  /* fp32 precision only.  `p` holds TWO pose sets back to back, p[2][B,Z,P]: p[0] = the poses the path is evaluated at, p[1] =
   * the poses whose relu ACTIVATION PATTERN the two RFF layers (rff.py:61) use: h = [pre(p[1]) > 0] * pre(p[0]).  With
   * p[1] = p[0] this is the plain path.  It exists for the second-order outer gradient of the meta-learning step
   * (jax.value_and_grad at pde_trainer.py:255 through jax.grad at :188): a Hessian-vector product is taken as a finite
   * difference of enf_xattn_bwd gradients along a latent direction, and freezing the pattern at the expansion point makes that
   * difference differentiate one linear branch of the relus -- exactly what reverse-over-reverse autodiff computes (relu'' = 0;
   * a plain finite difference would add the curvature concentrated at the kinks).  dp[B,Z,P] is the gradient w.r.t. p[0]. */
  ENF_FLAG_FROZEN_RELU = 16,
  /* The call is one LATENT SELF-ATTENTION step of the NeF (num_layers > 0: equivariant_cross_attention_nef.py:159-167, 223-226;
   * EquivariantCrossAttentionBlock with residual = True, project_heads = True, :44-67), not the cross-attention decode:
   *     out = gelu(a' + FFN(a' + out_proj(attn(x = p, p, LayerNorm(a')))))        a' = latent_stem(a) (or a, ENF_FLAG_NO_STEM)
   * The queries are the latent poses themselves (C must equal Z; `x` is ignored and may be NULL), the invariant is the
   * SELF-attention variant (get_sa_invariant: ENF_INV_PONITA means Ponita2D, 3 invariants), O must equal d and `out` is the
   * next hidden latent state [B,Z,d].  Weight leaves of EnfWeights with this flag: wo is (H*d, d), bo (d), the pointwise FFN
   * fb_* is d -> d -> d, m0_* / m1_* / m2_* are unused (may be NULL).  dp of enf_xattn_bwd carries the gradient through both roles
   * of the poses (query and latent).  Always runs the fp32 kernels (B*Z*Z pairs: <= 2 % of a decode call). */
  ENF_FLAG_SELF_BLOCK = 32,
  /* `a` is already the hidden latent state [B,Z,d] (the output of a self-attention step): latent_stem is skipped, L must
   * equal d, stem_w / stem_b are unused (may be NULL), da is [B,Z,d]. */
  ENF_FLAG_NO_STEM = 64,
  /* Training call that will also want the gradient w.r.t. the query coordinates x (enf_xattn_bwd_x): spatial derivatives of the
   * decoded field (gradient / Sobolev losses, PDE residuals), or a gradient that flows on into whatever computed x.  Set at
   * forward time: the workspace then also holds the cotangent of the per-query records, g_xi [B,C,8] (enf_xattn_workspace_bytes
   * grows by exactly that buffer).  Not with ENF_FLAG_FORWARD_ONLY, nor with ENF_FLAG_SELF_BLOCK (x is ignored there; dp
   * already carries the poses in both roles). */
  ENF_FLAG_GRAD_X = 128
};

enum EnfError {
  ENF_OK = 0,
  ENF_ERR_BAD_DESC = -1,        /* inconsistent / unsupported sizes                     */
  ENF_ERR_UNSUPPORTED = -2,     /* valid request the build does not implement           */
  ENF_ERR_NULL_POINTER = -3,
  ENF_ERR_WORKSPACE = -4,       /* workspace too small or misaligned                    */
  ENF_ERR_CUDA = -5,            /* a CUDA runtime call failed while enqueueing          */
  ENF_ERR_NO_DEVICE = -6,
  ENF_ERR_STATE = -7            /* bwd called on a workspace that holds no matching fwd */
};

/* Problem description.  Mirrors the constructor fields of EquivariantCrossAttentionNeF
 * (equivariant_cross_attention_nef.py:85-96) plus the call shapes. */
typedef struct EnfDesc {
  int32_t B;               /* fields (signals) in the call                                */
  int32_t C;               /* coordinate queries per field                                */
  int32_t Z;               /* latents per field                                           */
  int32_t d;               /* num_hidden  (16, 32, 64 or 128)                             */
  int32_t H;               /* num_heads   (1..4)                                          */
  int32_t L;               /* latent_dim                                                  */
  int32_t O;               /* num_out                                                     */
  int32_t Dx;              /* num_in (coordinate width)                                   */
  int32_t invariant_kind;  /* EnfInvariantKind                                            */
  int32_t use_window;      /* use_gaussian_window                                         */
  int32_t precision;       /* EnfPrecision                                                */
  int32_t flags;           /* EnfFlags (0 = training: the workspace keeps the state enf_xattn_bwd needs) */
  int32_t chunk_fields;    /* ENF_FLAG_RECOMPUTE: fields per backward chunk (0 = default: min(B, 4)); else ignored */
  int32_t reserved[3];     /* must be 0                                                   */
} EnfDesc;

/* The parameter leaves of nef.init(...)['params'] (Flax tree, SURVEY.md A.3), as device pointers.
 * Dense kernels are (in, out) row-major exactly as Flax stores them. */
typedef struct EnfWeights {
  const float *stem_w, *stem_b;                              /* latent_stem                  (L,d) (d)      */
  const float *ln_attn_g, *ln_attn_b;                        /* .../layer_norm_attn          (d) (d)        */
  const float *q_omega, *q_w1, *q_b1, *q_wf, *q_bf;          /* attn/invariant_embedding_query: coefficients (I,d/2), layers_0/linear, linear_final */
  const float *v_omega, *v_w1, *v_b1, *v_wf, *v_bf;          /* attn/invariant_embedding_value               */
  const float *wq, *bq, *wk, *bk, *wv, *bv;                  /* attn/inv_emb_to_q, a_to_k, a_to_v (d,Hd) (Hd) */
  const float *fv_w1, *fv_b1, *fv_g, *fv_beta, *fv_w2, *fv_b2; /* attn/inv_emb_to_v  Dense_0 (d,d), LayerNorm_0, Dense_1 (d,2Hd) */
  const float *mx_w1, *mx_b1, *mx_g, *mx_beta, *mx_w2, *mx_b2; /* attn/inv_emb_cond_mixer Dense_0 (d,d), LayerNorm_0, Dense_1 (d,d) */
  const float *wo, *bo;                                      /* attn/out_proj                (Hd,Hd) (Hd)   */
  const float *fb_w1, *fb_b1, *fb_g, *fb_beta, *fb_w2, *fb_b2; /* pointwise_ffn Dense_0, LayerNorm_0, Dense_1 (Hd,Hd) */
  const float *m0_w, *m0_b, *m1_w, *m1_b, *m2_w, *m2_b;      /* out_proj/layers_0 (Hd,d), layers_2 (d,d), layers_4 (d,O) */
} EnfWeights;

#define ENF_NUM_WEIGHT_LEAVES 46

/* Same leaves, writable: d(loss)/d(leaf).  q_omega / v_omega receive zeros (stop_gradient, rff.py:90). */
typedef struct EnfWeightGrads {
  float *stem_w, *stem_b;
  float *ln_attn_g, *ln_attn_b;
  float *q_omega, *q_w1, *q_b1, *q_wf, *q_bf;
  float *v_omega, *v_w1, *v_b1, *v_wf, *v_bf;
  float *wq, *bq, *wk, *bk, *wv, *bv;
  float *fv_w1, *fv_b1, *fv_g, *fv_beta, *fv_w2, *fv_b2;
  float *mx_w1, *mx_b1, *mx_g, *mx_beta, *mx_w2, *mx_b2;
  float *wo, *bo;
  float *fb_w1, *fb_b1, *fb_g, *fb_beta, *fb_w2, *fb_b2;
  float *m0_w, *m0_b, *m1_w, *m1_b, *m2_w, *m2_b;
} EnfWeightGrads;

typedef struct CUstream_st* enf_stream_t;   /* == cudaStream_t */

int enf_abi_version(void);

/* Width of the invariant (I) and of the RAW latent pose (num_z_pos_dims + num_z_ori_dims) for a kind;
 * negative on a bad kind.  Dx is the coordinate width (num_in). */
int enf_invariant_dim(int invariant_kind, int Dx);
int enf_pose_dim(int invariant_kind, int Dx);

/* Bytes of caller-provided scratch needed by enf_xattn_fwd / enf_xattn_bwd for this description
 * (0 on a bad description).  The same workspace must be passed to the bwd that follows a fwd:
 * it carries the forward state (softmax statistics, decode-MLP activations, per-latent folds). */
size_t enf_xattn_workspace_bytes(const EnfDesc* desc);

/* ENF_FLAG_RECOMPUTE: the largest chunk_fields (1..B) whose workspace fits in cap_bytes; 0 if even one field per chunk
 * does not fit (or on a bad description).  `desc->chunk_fields` is ignored. */
int enf_xattn_chunk_for_cap(const EnfDesc* desc, size_t cap_bytes);

/* Which kernels enf_xattn_fwd / enf_xattn_bwd run for this description (what bench.py labels its lines with):
 *   *fwd_tc, *bwd_tc = 1 when the fused pair forward / backward run on the tcgen05 kernels, 0 = fp32 FMA kernels.
 * Returns 0, or a negative EnfError on a bad description.  Either pointer may be NULL. */
int enf_xattn_dispatch(const EnfDesc* desc, int* fwd_tc, int* bwd_tc);

/* Forget the forward state kept for `workspace` (call before freeing or reusing the buffer for something else).
 * enf_xattn_bwd may be called any number of times after one enf_xattn_fwd (it does not consume the forward state). */
void enf_workspace_release(void* workspace);

/* out[B,C,O] = nef.apply(params, x, p, a, sigma)                       (replaces pde_trainer.py:184,478,537)
 *   x      [B,C,Dx]  with x_batch_stride = C*Dx, or ONE shared [C,Dx] grid with x_batch_stride = 0
 *   p      [B,Z,P]   raw latent poses (P = enf_pose_dim), a [B,Z,L], sigma [B,Z,1] (may be NULL iff !use_window)
 */
int enf_xattn_fwd(const EnfDesc* desc, const EnfWeights* w,
                  const float* x, int64_t x_batch_stride,
                  const float* p, const float* a, const float* sigma,
                  float* out, void* workspace, size_t workspace_bytes, enf_stream_t stream);   /* out: bf16 with ENF_FLAG_OUT_BF16 */

/* Reverse pass for cotangent d_out[B,C,O] of the enf_xattn_fwd call last issued on `workspace`
 * with the same arguments (x_batch_stride included; checked).   (replaces jax.grad at pde_trainer.py:188,255)
 * Repeatable: the forward state is not consumed, a second call with another cotangent gives that cotangent's gradients.
 *   dW      weight gradients (overwritten); NULL => latent gradients only (ode phase, pde_trainer.py:302)
 *   dp[B,Z,P], da[B,Z,L], dsigma[B,Z,1] overwritten (dsigma may be NULL; zeros if !use_window)
 */
int enf_xattn_bwd(const EnfDesc* desc, const EnfWeights* w,
                  const float* x, int64_t x_batch_stride,
                  const float* p, const float* a, const float* sigma,
                  const float* d_out, const EnfWeightGrads* dW,
                  float* dp, float* da, float* dsigma,
                  void* workspace, size_t workspace_bytes, enf_stream_t stream);

/* enf_xattn_bwd plus the gradient w.r.t. the query coordinates (the forward must have run with ENF_FLAG_GRAD_X):
 *   dx     overwritten; [B,C,Dx] when x_batch_stride == C*Dx, [C,Dx] for one shared grid (x_batch_stride == 0): then dx is the
 *          sum over the B fields.  Required (non-NULL) on a description with ENF_FLAG_GRAD_X; NULL is accepted only without
 *          that flag (then this is enf_xattn_bwd), a non-NULL dx without it returns ENF_ERR_STATE.
 * enf_xattn_bwd on an ENF_FLAG_GRAD_X workspace computes everything but dx, at the cost of a backward without the flag.
 * Like x itself, dx is reached only through the per-query records: the op is once differentiable in x as in everything else. */
int enf_xattn_bwd_x(const EnfDesc* desc, const EnfWeights* w,
                    const float* x, int64_t x_batch_stride,
                    const float* p, const float* a, const float* sigma,
                    const float* d_out, const EnfWeightGrads* dW,
                    float* dp, float* da, float* dsigma, float* dx,
                    void* workspace, size_t workspace_bytes, enf_stream_t stream);

/* Number of kernels of this library enqueued by the last fwd / bwd call of the calling thread. */
int enf_last_launch_count(void);

/* Measurement hook (bench.py).  While enabled, a CUDA event pair is recorded on the call's stream around the
 * fused pair kernel of every fwd (which = 0) / bwd (which = 1), in a ring of 256.  enf_profile_collect waits
 * for those kernels, writes up to max_out device times in milliseconds (oldest first), resets the ring and
 * returns how many it wrote (-1 on error).  Not thread-safe; off by default. */
int enf_profile_enable(int on);
int enf_profile_collect(int which, float* ms_out, int max_out);

/* Thread-local description of the last error returned on this thread ("" if none). */
const char* enf_last_error(void);

/* Test/diagnostic hook: byte offset and element count of a named internal workspace buffer
 * (e.g. "xi", "lam", "U", "W3", "nbar", "lse"); returns -1 if unknown. */
int64_t enf_debug_ws_offset(const EnfDesc* desc, const char* name, int64_t* num_floats);

/* Test hook: one 128-row tcgen05 tile GEMM with bf16 operands (D = 64 or 128 features), pinning the
 * shared-memory descriptor / swizzle conventions of the tensor-core kernels on hardware.
 *   mode 0: out[r][n] = sum_k X[r][k] Y[n][k];  mode 1: out[r][k] = sum_n X[r][n] Y[n][k];
 *   mode 2: out[i][j] = sum_r X[r][i] Y[r][j].   X, Y, out: device float32 [128][D]; scratch >= D*D*2 bytes. */
int enf_debug_tc_gemm(int mode, int D, const float* X, const float* Y, float* out, void* scratch, enf_stream_t stream);

/* Test hook: one stage GEMM  C[M,N] (+)= A[M,K] B[K,N] (+bias) (*gelu'(aux)), optional gelu_out = gelu(C), through the
 * library's own dispatcher (use_tc != 0: the tf32 tcgen05/TMA kernels when the shape qualifies, else the fp32 kernel).
 * All matrices are device float32 with explicit (row, column) strides in elements.  B_lo (nullable) = B - trunc_tf32(B)
 * with B's strides: required by the tensor-core product kernel (3-term split).  Returns the number of kernels
 * launched, or a negative error code. */
int enf_debug_gemm(int use_tc, int M, int N, int K, const float* A, int64_t a_rs, int64_t a_cs, const float* B, int64_t b_rs,
                   int64_t b_cs, const float* B_lo, float* C, int64_t c_rs, const float* bias, const float* aux, float* gelu_out,
                   int accumulate, enf_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* ENF_B200_H_ */
