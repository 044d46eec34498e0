// Shared definitions for the ENF B200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#include "../../include/enf_b200.h"

#define ENF_F_XI 8    // width of the per-query feature record xi
#define ENF_R_LAM 7   // rows of the per-latent pose record Lam (<= 6 invariant rows + 1 window row)
#define ENF_LAM_SIZE (ENF_R_LAM * ENF_F_XI)

enum { ENF_ROW_DOT = 0, ENF_ROW_SQDIST = 1, ENF_ROW_SQDIST_SQRT = 2 };
enum { ENF_WIN_NONE = 0, ENF_WIN_NP = 1, ENF_WIN_PER = 2, ENF_WIN_SPH = 3 };

// How the hot kernels evaluate invariants: u_r = post_r(row_r(Lam[z], xi[c])) (DESIGN.md "Invariant records").
struct EnfRecordLayout {
  int I;          // invariant width
  int row_kind;   // kind of the invariant rows (all rows of one invariant share it)
  int win_kind;   // ENF_WIN_*
  int win_row;    // row of Lam holding the window's record (== I), or -1 when the window reads u[0]
  int nsq;        // components compared by SQDIST rows
};
// ... and the raw pose width, which only the record producers read (enf_stages.cu)
struct EnfInvariantLayout : EnfRecordLayout { int P; };

__host__ __device__ inline EnfInvariantLayout enf_record_layout(int kind, int Dx, int use_window) {
  EnfInvariantLayout r;
  r.row_kind = ENF_ROW_DOT; r.nsq = Dx; r.win_row = -1;
  int win = ENF_WIN_NP;
  switch (kind) {
    case ENF_INV_REL_POS: r.I = Dx; r.P = Dx; break;
    case ENF_INV_NORM_REL_POS: r.I = 1; r.P = Dx; r.row_kind = ENF_ROW_SQDIST_SQRT; break;
    case ENF_INV_ABS_POS: r.I = Dx; r.P = Dx; break;
    case ENF_INV_REL_POS_PERIODIC: r.I = 4; r.P = 2; win = ENF_WIN_PER; break;
    case ENF_INV_PONITA: r.I = 2; r.P = 3; r.nsq = 2; break;
    case ENF_INV_POLAR_PERIODIC: r.I = 1; r.P = 2; win = ENF_WIN_SPH; break;
    case ENF_INV_LATITUDE_PERIODIC: r.I = 4; r.P = 2; win = ENF_WIN_SPH; break;
    case ENF_INV_BALL: r.I = 5; r.P = 4; win = ENF_WIN_SPH; break;
    case ENF_INV_BALL_LAT: r.I = 6; r.P = 4; win = ENF_WIN_SPH; break;
    default: r.I = -1; r.P = -1; break;
  }
  r.win_kind = use_window ? win : ENF_WIN_NONE;
  if (r.win_kind == ENF_WIN_NP) r.win_row = r.I;
  if (r.win_kind == ENF_WIN_SPH && kind != ENF_INV_POLAR_PERIODIC) r.win_row = r.I;
  return r;
}

// ---- the record algebra of one (query, latent) pair, shared by every pair kernel (fp32, tensor-core, latent ODE) ---------
// lam: the latent's record Lam [ENF_R_LAM][ENF_F_XI]; x / xi: the query's record [ENF_F_XI].  SQDIST rows compare nsq <= 3 components.
struct EnfPairRecord { float u[6]; float w; float c; };   // invariants, window value, raw cosine (spherical windows)

// invariant row r of one pair: u_r = post(row_r(Lam, xi))
__device__ __forceinline__ float record_row(const EnfRecordLayout& rl, const float* lam, const float* x, int r) {
  const float* L = lam + r * ENF_F_XI;
  float v = 0.f;
  if (rl.row_kind == ENF_ROW_DOT) {
#pragma unroll
    for (int f = 0; f < 8; ++f) v = fmaf(L[f], x[f], v);
  } else {
#pragma unroll
    for (int f = 0; f < 3; ++f) if (f < rl.nsq) { float dl = L[f] - x[f]; v = fmaf(dl, dl, v); }
    if (rl.row_kind == ENF_ROW_SQDIST_SQRT) v = sqrtf(v);
  }
  return v;
}

// window value w (and the raw cosine c of the spherical windows) from the invariants it reads (u0, u1) and the window row.
// FAST_EXP: __expf on the tensor-core path (its 16-bit operands dominate the error), expf on the fp32 path (the accurate one).
template <bool FAST_EXP>
__device__ __forceinline__ void record_window(const EnfRecordLayout& rl, const float* lam, const float* x, float sigma, float u0, float u1,
                                              float& w, float& c) {
  w = 0.f; c = 0.f;
  if (rl.win_kind == ENF_WIN_NONE) return;
  const float* L = lam + rl.I * ENF_F_XI;
  float inv_s2 = 1.f / (sigma * sigma);
  if (rl.win_kind == ENF_WIN_NP) {
    float v = 0.f;
#pragma unroll
    for (int f = 0; f < 3; ++f) if (f < rl.nsq) { float dl = L[f] - x[f]; v = fmaf(dl, dl, v); }
    w = -v * inv_s2;
  } else if (rl.win_kind == ENF_WIN_PER) {
    w = fmaf(u0, u0, u1 * u1) * inv_s2;
  } else {
    c = u0;
    if (rl.win_row >= 0) {
      c = 0.f;
#pragma unroll
      for (int f = 0; f < 8; ++f) c = fmaf(L[f], x[f], c);
    }
    float cl = fminf(fmaxf(c, -1.f + 1e-6f), 1.f - 1e-6f);
    float ac = acosf(cl);
    w = FAST_EXP ? __expf(-ac * ac * 0.5f * inv_s2) : expf(-ac * ac * 0.5f * inv_s2);
  }
}
// the invariants u0, u1 that record_window reads, for a caller that holds none of them (0 where the window does not read them)
__device__ __forceinline__ void record_window_rows(const EnfRecordLayout& rl, const float* lam, const float* x, float& u0, float& u1) {
  u0 = 0.f; u1 = 0.f;
  if (rl.win_kind == ENF_WIN_PER) { u0 = record_row(rl, lam, x, 0); u1 = record_row(rl, lam, x, 1); }
  else if (rl.win_kind == ENF_WIN_SPH && rl.win_row < 0) u0 = record_row(rl, lam, x, 0);
}

template <bool FAST_EXP>
__device__ __forceinline__ EnfPairRecord pair_record(const EnfRecordLayout& rl, const float* lam, const float* xi, float sigma) {
  EnfPairRecord r;
  float x[8];
#pragma unroll
  for (int f = 0; f < 8; ++f) x[f] = xi[f];
#pragma unroll
  for (int i = 0; i < 6; ++i) r.u[i] = i < rl.I ? record_row(rl, lam, x, i) : 0.f;
  record_window<FAST_EXP>(rl, lam, x, sigma, r.u[0], r.u[1], r.w, r.c);
  return r;
}

// cotangent of the squared distance v of a SQDIST_SQRT row u = sqrt(v) from the cotangent du of u
__device__ __forceinline__ float record_sqrt_adjoint(float du, float u) { return u > 0.f ? du / (2.f * u) : 0.f; }

// cotangents of one pair's record rows dq (dq[I]: the window row) and of sigma from those of the invariants (du; the periodic
// window and the spherical window without a window row add to du[0..1]) and of the window value (dw)
__device__ __forceinline__ void record_adjoint(const EnfRecordLayout& rl, const EnfPairRecord& rec, float (&du)[6], float dw, float sigma,
                                               float (&dq)[ENF_R_LAM], float& dsg) {
#pragma unroll
  for (int r = 0; r < ENF_R_LAM; ++r) dq[r] = 0.f;
  dsg = 0.f;
  if (rl.win_kind != ENF_WIN_NONE) {
    const float inv_s2 = 1.f / (sigma * sigma);
    if (rl.win_kind == ENF_WIN_NP) {
      dq[rl.I] = -dw * inv_s2;
      dsg = dw * (-2.f * rec.w / sigma);
    } else if (rl.win_kind == ENF_WIN_PER) {
      du[0] += dw * 2.f * rec.u[0] * inv_s2;
      du[1] += dw * 2.f * rec.u[1] * inv_s2;
      dsg = dw * (-2.f * rec.w / sigma);
    } else {
      float cl = fminf(fmaxf(rec.c, -1.f + 1e-6f), 1.f - 1e-6f);
      float ac = acosf(cl);
      float dc = (rec.c > -1.f + 1e-6f && rec.c < 1.f - 1e-6f) ? dw * rec.w * ac * inv_s2 * rsqrtf(1.f - cl * cl) : 0.f;
      if (rl.win_row >= 0) dq[rl.I] = dc; else du[0] += dc;
      dsg = dw * rec.w * ac * ac * inv_s2 / sigma;
    }
  }
#pragma unroll
  for (int r = 0; r < 6; ++r) {
    if (r < rl.I) {
      if (rl.row_kind == ENF_ROW_SQDIST_SQRT) dq[r] = record_sqrt_adjoint(du[r], rec.u[r]);
      else dq[r] = du[r];
    }
  }
}

// g[k] += d xi[f] = sum_r dq_r d row_r / d xi[f] for the half f = 4 half + k, k < 4 of the query record: DOT rows are bilinear in
// (Lam, xi); squared-distance rows (and the non-periodic window row) are sum_{f < nsq} (Lam_f - xi_f)^2, so they only reach half 0
__device__ __forceinline__ void record_xi_cotangent(const EnfRecordLayout& rl, const float* lam, const float* xi, const float (&dq)[ENF_R_LAM],
                                                    int half, float* g) {
  const float* Lh = lam + 4 * half;
#pragma unroll
  for (int r = 0; r < ENF_R_LAM; ++r) {
    if (r < rl.I || (r == rl.I && rl.win_row >= 0)) {
      const float* L = Lh + r * ENF_F_XI;
      const bool sq = r < rl.I ? (rl.row_kind != ENF_ROW_DOT) : (rl.win_kind == ENF_WIN_NP);
      if (!sq) {
#pragma unroll
        for (int k = 0; k < 4; ++k) g[k] = fmaf(dq[r], L[k], g[k]);
      } else if (half == 0) {
#pragma unroll
        for (int k = 0; k < 3; ++k) if (k < rl.nsq) g[k] = fmaf(-2.f * dq[r], L[k] - xi[k], g[k]);
      }
    }
  }
}

// jax.nn.gelu(approximate=True)
__device__ __forceinline__ float enf_gelu(float x) {
  const float c = 0.7978845608028654f;
  return 0.5f * x * (1.0f + tanhf(c * (x + 0.044715f * x * x * x)));
}
__device__ __forceinline__ float enf_gelu_grad(float x) {
  const float c = 0.7978845608028654f;
  float x2 = x * x;
  float t = tanhf(c * (x + 0.044715f * x * x2));
  return 0.5f * (1.0f + t) + 0.5f * x * (1.0f - t * t) * c * (1.0f + 3.0f * 0.044715f * x2);
}

// round-to-nearest to the 10-bit tf32 mantissa: what producers store for operands of the tf32 GEMMs (enf_gemm_tc.cu)
__device__ __forceinline__ float enf_round_tf32(float x) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
  return __uint_as_float(u);
}
__device__ __forceinline__ float enf_maybe_round(float x, int rnd) { return rnd ? enf_round_tf32(x) : x; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---- generic strided GEMM (enf_gemm.cu) ------------------------------------------------------
struct EnfMat {            // a strided 2-D view with an optional batch stride
  const float* p;
  int64_t rs, cs, bs;
};
static inline EnfMat enf_mat(const float* p, int64_t rs, int64_t cs = 1, int64_t bs = 0) {
  EnfMat m; m.p = p; m.rs = rs; m.cs = cs; m.bs = bs; return m;
}
struct EnfGemmOpts {
  int batch = 1;
  const float* bias = nullptr;      // [N], added once
  int64_t bias_bs = 0;              // batch stride of bias
  int act_a = 0;                    // 1: A elements pass through gelu on load
  const float* mul_gelu_grad = nullptr;  // epilogue: result *= gelu'(aux[m,n]) (aux has C's strides)
  int accumulate = 0;               // 1: atomicAdd into C (C must hold the running sum); enables split-K
  float alpha = 1.0f;
  float* gelu_out = nullptr;        // optional second output gelu(C), laid out like C
  int round_out = 0;                // 1: store C (and gelu_out) rounded to tf32
  int tc = 0;                       // 1: use the tf32 tensor-core kernels (enf_gemm_tc.cu) when the shape allows
  const float* b_lo = nullptr;      // tensor-core path: B - trunc_tf32(B), same strides as B (3-term split product)
};
// C[M,N] (+)= alpha * act(A)[M,K] * B[K,N] (+ bias) (* gelu'(aux)); returns number of kernels launched.
int enf_gemm(cudaStream_t st, int M, int N, int K, EnfMat A, EnfMat B, EnfMat C, const EnfGemmOpts& o);
// several small independent products (batch 1, no split-K, not tensor-core) in one launch; returns the number of launches
struct EnfGemmProblem { int M, N, K; EnfMat A, B, C; EnfGemmOpts o; };
bool enf_gemm_groupable(int M, int N, int K, const EnfGemmOpts& o);
int enf_gemm_group(cudaStream_t st, int n, const EnfGemmProblem* p);
// tf32 tensor-core path: 1 = launched, 0 = shape not taken (use the fp32 kernel), -1 = configuration error
int enf_gemm_tc(cudaStream_t st, int M, int N, int K, EnfMat A, EnfMat B, EnfMat C, const EnfGemmOpts& o);
// dst[i] = src[i] - trunc_tf32(src[i]) for up to 8 (src, dst, n) triples in one launch (the B_lo operands)
struct EnfSplitList { const float* src[8]; float* dst[8]; int n[8]; int count; };
int enf_launch_split_lo(cudaStream_t st, const EnfSplitList& l);

// ---- small stage kernels (enf_stages.cu) -------------------------------------------------------
int enf_launch_rowscale(cudaStream_t st, const float* W, const float* g, float* out, int rows, int cols);
int enf_launch_colsum(cudaStream_t st, const float* G, int64_t M, int N, int64_t ld, float* out, const float* mul, int64_t ld_mul);
// decode MLP's last layer (d -> O, O <= 4): out = act(A) W + b ; dX = (dO W^T) gelu'(pre) ; dW += act(A)^T dO, db += colsum(dO)
bool enf_thin_supported(int d, int O);
int enf_launch_thin_out(cudaStream_t st, const float* A, const float* W, const float* b, float* out, int64_t M, int d, int O, int act_a,
                        int out_bf16 = 0);     // out_bf16: `out` is a bfloat16 buffer (ENF_FLAG_OUT_BF16)
int enf_launch_thin_dgrad(cudaStream_t st, const float* dO, const float* W, const float* pre, float* dX, int64_t M, int d, int O);
int enf_launch_thin_wgrad(cudaStream_t st, const float* A, const float* dO, float* dW, float* db, int64_t M, int d, int O, int act_a);
int enf_launch_ln_fwd(cudaStream_t st, const float* in, int64_t M, int N, const float* g, const float* b,
                      float* out_core, float* out_affine, float* rstd, int gelu_in, int round_affine = 0);
int enf_launch_ln_bwd(cudaStream_t st, const float* dy, const float* core, const float* rstd, const float* g,
                      const float* pre, int64_t M, int N, float* dx, float* dg, float* db, int gelu_in, int round_dx = 0,
                      int fast_gelu = 0);
int enf_launch_query_features(cudaStream_t st, const EnfDesc& d, const float* x, int64_t xbs, int Bx, float* xi);
int enf_launch_latent_record(cudaStream_t st, const EnfDesc& d, const float* p, float* lam);
int enf_launch_latent_record_bwd(cudaStream_t st, const EnfDesc& d, const float* p, const float* dlam, float* dp);
// poses used as queries (latent ODE model: invariant(p, p)); self-attention variants of the invariants (ENF_INV_PONITA = Ponita2D, I = 3)
int enf_launch_pose_features(cudaStream_t st, int kind, int Dx, int P, int64_t total, const float* p, float* xi);
int enf_launch_pose_features_bwd(cudaStream_t st, int kind, int Dx, int P, int64_t total, const float* p, const float* dxi, float* dp);   // dp +=
// decode queries: d(record) [B,C,8] -> dx [Bx,C,Dx] (overwritten; Bx = 1: a shared grid, summed over the B fields)
int enf_launch_coord_features_bwd(cudaStream_t st, const EnfDesc& d, const float* x, int Bx, const float* dxi, float* dx);
int enf_launch_pose_record(cudaStream_t st, int kind, int Dx, int P, int I, int64_t total, const float* p, float* lam);
int enf_launch_pose_record_bwd(cudaStream_t st, int kind, int Dx, int P, int I, int win_kind, int64_t total, const float* p, const float* dlam, float* dp);   // dp =
int enf_launch_weff(cudaStream_t st, const EnfDesc& d, const float* W2g, const float* b2g, const float* v0,
                    float* Weff, float* beff, int round_weff = 0);
int enf_launch_weff_bwd(cudaStream_t st, const EnfDesc& d, const float* W2g, const float* b2g, const float* v0,
                        const float* dWeff, const float* dbeff, float* dW2g, float* db2g, float* dv0);
int enf_launch_add_outer(cudaStream_t st, float* C, int64_t ldc, const float* u, const float* v, int M, int N);
int enf_launch_rowdot(cudaStream_t st, const float* A, const float* Bm, float* out, int rows, int cols);
int enf_launch_mul_rows(cudaStream_t st, float* out, const float* A, const float* g, int rows, int cols,
                        const float* add_outer_u, const float* add_outer_v);
int enf_launch_transpose(cudaStream_t st, const float* in, float* out, int rows, int cols, int batch);
// out = a + b ; pre = a + b, out = gelu(pre) ; out (+)= g * gelu'(pre)
int enf_launch_add(cudaStream_t st, float* out, const float* a, const float* b, int64_t n);
int enf_launch_add_gelu(cudaStream_t st, float* pre, float* out, const float* a, const float* b, int64_t n);
int enf_launch_mul_gelu_grad(cudaStream_t st, float* out, const float* g, const float* pre, int64_t n);

int enf_launch_weight_image(cudaStream_t st, const float* Wt, void* img, float* cw, int N, int K, int batch, int residual = 0);
// image of W^T built from the untransposed W [batch][K][N] (no fp32 transpose pass)
int enf_launch_weight_image_T(cudaStream_t st, const float* W, void* img, int N, int K, int batch);

// ---- fused pair kernels (enf_pairs_simt.cu) ------------------------------------------------------
struct EnfPairParams {
  int B, C, Z, H;
  EnfRecordLayout rec;
  const float* xi;  int64_t xi_bs;           // [Bx, C, 8]
  const float* lam;                          // [B, Z, 7, 8]
  const float* lam_mask;                     // frozen-relu mode (ENF_FLAG_FROZEN_RELU): record of the mask poses, else null
  const float* sigma;                        // [B, Z] or null
  const float* q_omega; const float* v_omega;  // [I, d/2]
  const float* q_w1; const float* q_b1;      // [d, d], [d]
  const float* v_w1; const float* v_b1;
  const float* Wp; const float* bp;          // folded linear_final_v o FFN_v.Dense_0
  const float* U; const float* kappa;        // [B,Z,H,d], [B,Z,H]
  const float* W3; const float* b3;          // [B,Z,H,d,d], [B,Z,H,d]
  float* nbar; float* lse;                   // [B,C,H,d], [B,C,H]
  // backward only
  const float* q_w1T; const float* v_w1T; const float* WpT; const float* W3T;   // transposed copies
  const float* dnbar;                        // [B,C,H,d]
  const float* slog;                         // [B,Z,C,H] logits saved by the tensor-core forward (or null: recompute)
  float* g_q_w1; float* g_q_b1; float* g_v_w1; float* g_v_b1; float* g_Wp; float* g_bp;   // accumulated (atomics)
  float* g_W3; float* g_b3; float* g_U; float* g_kappa; float* g_lam; float* g_sigma;      // per-latent, accumulated
  float* g_xi;                               // [B,C,8] cotangent of the query records (self-attention blocks, ENF_FLAG_GRAD_X), else null
};
int enf_launch_pairs_fwd_simt(cudaStream_t st, int d, const EnfPairParams& p);
int enf_launch_pairs_bwd_simt(cudaStream_t st, int d, const EnfPairParams& p);

// ---- tensor-core pair kernels (enf_pairs_tc.cu) ----------------------------------------------------
struct EnfPairTcParams {
  int B, C, Z;
  EnfRecordLayout rec;
  const float* xi;  int64_t xi_bs;
  const float* lam; const float* sigma;
  const float* q_omega; const float* v_omega;
  const float* q_b1; const float* v_b1; const float* bp;
  const uint8_t* img_q_w1; const uint8_t* img_v_w1; const uint8_t* img_Wp;   // bf16 operand images of W^T ([n][k])
  const uint8_t* img_W3;                     // [B*Z*H] images of W3^T
  const float* U; const float* kappa; const float* b3;
  float* nbar; float* lse; float* slog;      // slog [B,Z,C,H]: logits incl. window (saved for the backward), may be null
  uint8_t* that_img;                         // [B,Z,ceil(C/128)] operand images (128 rows x d, fp16, swizzled) of that = LN(gelu(.)),
                                             // stashed for backward kernel A; may be null (forward only / SIMT backward)
  uint4* dgr;                                // gelu'(tpre) of the same layer, fp16, in backward kernel B's load order (the chunked
                                             // order of dthat below); stashed together with that_img, null when that is
  float* trstd;                              // [B,Z,ceil(C/128)*128] reciprocal standard deviation of that LayerNorm (with dgr)
};
bool enf_pairs_fwd_tc_supported(int d, int H);
int enf_launch_pairs_fwd_tc(cudaStream_t st, int d, int H, const EnfPairTcParams& p);

struct __half;
struct EnfPairTcBwdParams {
  int B, C, Z;
  EnfRecordLayout rec;
  const float* xi;  int64_t xi_bs;
  const float* lam; const float* sigma;
  const float* q_omega; const float* v_omega;
  const float* q_b1; const float* v_b1; const float* bp;
  const uint8_t* img_q_w1; const uint8_t* img_v_w1; const uint8_t* img_Wp; const uint8_t* img_W3;
  const uint8_t* img_q_w1_lo; const uint8_t* img_v_w1_lo;   // images of W - round16(W) (two-term split of the relu layers)
  const float* U; const float* b3;
  const float* slog; const float* lse; const float* nbar;   // forward state
  const uint8_t* that_img;                   // [B,Z,ceil(C/128)] that operand images stashed by the forward
  const uint4* dgr;                          // gelu'(tpre), fp16, chunked order of dthat (stashed by the forward for kernel B)
  const float* trstd;                        // [B,Z,ceil(C/128)*128] rstd of the LayerNorm producing that (stashed by the forward)
  const float* dnbar;                        // [B,C,H,d] cotangent of nbar
  float* Dg;                                 // [B,C,H]   dnbar16 . nbar              (written by the prep kernels)
  float* gmax;                               // [1]       max |dnbar| (zero-initialised; written by the prep kernels)
  uint4* dnb16;                              // scaled fp16 copy of dnbar in kernel A's load order:
                                             //   [B][C/128][H][4 column quarters][4 chunks][128 rows] x 8 halves (prep kernels)
  __half* dthat;                             // scaled cotangent of that (A -> B), same chunked order:
                                             //   [B,Z][C/128][4 column quarters][4 chunks][128 rows] x 8 halves
  float* ds;                                 // [B,Z,C,H] scaled cotangent of logits  (A -> C)
  float* duv;                                // [B,Z,C,8] scaled cotangent of the invariants through the value path (B -> C)
  float* g_W3; float* g_b3;                  // per-latent outputs of A
  float* g_q_w1; float* g_q_b1; float* g_v_w1; float* g_v_b1; float* g_Wp; float* g_bp;   // shared-weight grads (atomics)
  float* g_U; float* g_kappa; float* g_lam; float* g_sigma;                                // per-latent outputs of B
  float* g_xi;                               // [B,C,8] cotangent of the query records, accumulated by C (ENF_FLAG_GRAD_X), else null
};
bool enf_pairs_bwd_tc_supported(int d, int H);
// prep (once per backward, whole batch): gradient scale, fp16 cotangent of nbar, Dg;  main: kernels A, B, C on p.B fields
int enf_launch_pairs_bwd_tc_prep(cudaStream_t st, int d, int H, const EnfPairTcBwdParams& p);
int enf_launch_pairs_bwd_tc_main(cudaStream_t st, int d, int H, const EnfPairTcBwdParams& p);
int enf_launch_pairs_bwd_tc_v(cudaStream_t st, int d, const EnfPairTcBwdParams& p);          // kernel B (value path, bottom), called by the above
int enf_launch_pairs_bwd_tc_q(cudaStream_t st, int d, int H, const EnfPairTcBwdParams& p);   // kernel C (query path), called by the above
