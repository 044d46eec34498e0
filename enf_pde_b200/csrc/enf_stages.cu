// Small per-query (X), per-latent (L) and per-weight (W) stage kernels around the fused pair
// kernels: invariant records, LayerNorm rows, FiLM effective weights, reductions.  All fp32.
#include <cuda_bf16.h>

#include "enf_common.cuh"

namespace {

__device__ __forceinline__ void sph_unit(float phi, float th, float* o) {
  float sp, cp, st, ct;
  sincosf(phi, &sp, &cp);
  sincosf(th, &st, &ct);
  o[0] = st * cp; o[1] = st * sp; o[2] = ct;
}
// derivatives of the unit vector wrt (phi, theta)
__device__ __forceinline__ void sph_unit_grad(float phi, float th, float* dphi, float* dth) {
  float sp, cp, st, ct;
  sincosf(phi, &sp, &cp);
  sincosf(th, &st, &ct);
  dphi[0] = -st * sp; dphi[1] = st * cp; dphi[2] = 0.f;
  dth[0] = ct * cp; dth[1] = ct * sp; dth[2] = -st;
}

// ---- X: per-query feature record xi (SURVEY A.2; one record serves every latent) ----------------
// `xrs`: floats between consecutive rows of x (Dx for coordinate grids; the raw pose width when the "queries" are the latent
// poses themselves: latent ODE model / self-attention).  `sa`: self-attention variant of the invariant (get_sa_invariant:
// only `ponita` differs, Ponita2D reads the query's orientation angle xr[2] too).
__global__ void query_features_kernel(int kind, int Dx, int C, int64_t total, const float* __restrict__ x,
                                      int64_t xbs, float* __restrict__ xi, int xrs, int sa) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  int64_t b = t / C, c = t % C;
  const float* xr = x + b * xbs + c * xrs;
  float o[ENF_F_XI];
#pragma unroll
  for (int f = 0; f < ENF_F_XI; ++f) o[f] = 0.f;
  switch (kind) {
    case ENF_INV_REL_POS: case ENF_INV_NORM_REL_POS: case ENF_INV_ABS_POS:
      for (int i = 0; i < Dx; ++i) o[i] = xr[i];
      o[Dx] = 1.f;
      break;
    case ENF_INV_REL_POS_PERIODIC:
      sincospif(xr[0], &o[1], &o[0]);
      sincospif(xr[1], &o[3], &o[2]);
      break;
    case ENF_INV_PONITA:
      o[0] = xr[0]; o[1] = xr[1]; o[2] = 1.f;
      if (sa) sincosf(xr[2], &o[4], &o[3]);         // Ponita2D (ponita.py:84): x_ori . p_ori
      break;
    case ENF_INV_POLAR_PERIODIC:
      sph_unit(xr[0], xr[1], o);
      break;
    case ENF_INV_LATITUDE_PERIODIC: case ENF_INV_BALL_LAT:
      o[0] = xr[1];
      sincosf(xr[0], &o[2], &o[1]);
      o[3] = 1.f;
      sph_unit(xr[0], xr[1], o + 4);
      if (kind == ENF_INV_BALL_LAT) o[7] = xr[2];
      break;
    case ENF_INV_BALL:
      sph_unit(xr[0], xr[1], o);
      o[3] = xr[2]; o[4] = 1.f;
      break;
  }
  float4* dst = reinterpret_cast<float4*>(xi + t * ENF_F_XI);
  dst[0] = make_float4(o[0], o[1], o[2], o[3]);
  dst[1] = make_float4(o[4], o[5], o[6], o[7]);
}

// ---- L: per-latent pose record Lam (raw poses; the ponita cos/sin embed of nef.py:214-217 is folded in)
__global__ void latent_record_kernel(int kind, int Dx, int P, int I, int64_t total, const float* __restrict__ p,
                                     float* __restrict__ lam, int sa) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const float* pr = p + t * P;
  float L[ENF_R_LAM][ENF_F_XI];
#pragma unroll
  for (int r = 0; r < ENF_R_LAM; ++r)
#pragma unroll
    for (int f = 0; f < ENF_F_XI; ++f) L[r][f] = 0.f;
  const int W = I;
  switch (kind) {
    case ENF_INV_REL_POS:
      for (int i = 0; i < Dx; ++i) { L[i][i] = 1.f; L[i][Dx] = -pr[i]; L[W][i] = pr[i]; }
      break;
    case ENF_INV_NORM_REL_POS:
      for (int i = 0; i < Dx; ++i) { L[0][i] = pr[i]; L[W][i] = pr[i]; }
      break;
    case ENF_INV_ABS_POS:
      for (int i = 0; i < Dx; ++i) { L[i][i] = 1.f; L[W][i] = pr[i]; }
      break;
    case ENF_INV_REL_POS_PERIODIC:
      for (int i = 0; i < 2; ++i) {
        float s, c; sincospif(pr[i], &s, &c);
        L[i][2 * i] = c; L[i][2 * i + 1] = s;
        L[2 + i][2 * i] = s; L[2 + i][2 * i + 1] = -c;
      }
      break;
    case ENF_INV_PONITA: {
      float o0, o1; sincosf(pr[2], &o1, &o0);
      L[0][0] = o0; L[0][1] = o1; L[0][2] = -(pr[0] * o0 + pr[1] * o1);
      L[1][0] = -o1; L[1][1] = o0; L[1][2] = pr[0] * o1 - pr[1] * o0;
      if (sa) { L[2][3] = o0; L[2][4] = o1; }        // Ponita2D's third invariant (then I = 3 and the window row is row 3)
      L[W][0] = pr[0]; L[W][1] = pr[1];
    } break;
    case ENF_INV_POLAR_PERIODIC:
      sph_unit(pr[0], pr[1], L[0]);
      break;
    case ENF_INV_LATITUDE_PERIODIC: case ENF_INV_BALL_LAT: {
      float s, c; sincosf(pr[0], &s, &c);
      L[0][0] = 1.f;
      L[1][3] = pr[1];
      L[2][1] = c; L[2][2] = s;
      L[3][1] = -s; L[3][2] = c;
      if (kind == ENF_INV_BALL_LAT) { L[4][7] = 1.f; L[5][3] = pr[3]; }
      sph_unit(pr[0], pr[1], &L[W][4]);
    } break;
    case ENF_INV_BALL: {
      float sa, ca, sb, cb, sg, cg;
      sincosf(pr[0], &sa, &ca); sincosf(pr[1], &sb, &cb); sincosf(pr[2], &sg, &cg);
      L[0][0] = ca * cb; L[0][1] = ca * sb * sg - sa * cg; L[0][2] = ca * sb * cg + sa * sg;
      L[1][0] = sa * cb; L[1][1] = sa * sb * sg + ca * cg; L[1][2] = sa * sb * cg - ca * sg;
      L[2][0] = -sb;     L[2][1] = cb * sg;                L[2][2] = cb * cg;
      L[3][3] = 1.f;
      L[4][4] = pr[3];
      sph_unit(pr[0], pr[1], L[W]);
    } break;
  }
  float* dst = lam + t * ENF_LAM_SIZE;
#pragma unroll
  for (int r = 0; r < ENF_R_LAM; ++r)
#pragma unroll
    for (int f = 0; f < ENF_F_XI; ++f) dst[r * ENF_F_XI + f] = L[r][f];
}

// acc[r][f] = sum over queries of dq_r * xi_f (what the pair backward accumulates) -> d(raw pose)
__global__ void latent_record_bwd_kernel(int kind, int Dx, int P, int I, int win_kind, int64_t total,
                                         const float* __restrict__ p, const float* __restrict__ acc_all,
                                         float* __restrict__ dp, int sa) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const float* pr = p + t * P;
  const float* A = acc_all + t * ENF_LAM_SIZE;
#define ACC(r, f) A[(r) * ENF_F_XI + (f)]
  float g[4] = {0.f, 0.f, 0.f, 0.f};
  const int W = I;
  const bool np = (win_kind == ENF_WIN_NP);
  switch (kind) {
    case ENF_INV_REL_POS:
      for (int i = 0; i < Dx; ++i) {
        g[i] = -ACC(i, Dx);
        if (np) g[i] += 2.f * (pr[i] * ACC(W, Dx) - ACC(W, i));
      }
      break;
    case ENF_INV_NORM_REL_POS:
      for (int i = 0; i < Dx; ++i) {
        g[i] = 2.f * (pr[i] * ACC(0, Dx) - ACC(0, i));
        if (np) g[i] += 2.f * (pr[i] * ACC(W, Dx) - ACC(W, i));
      }
      break;
    case ENF_INV_ABS_POS:
      for (int i = 0; i < Dx; ++i) if (np) g[i] = 2.f * (pr[i] * ACC(W, Dx) - ACC(W, i));
      break;
    case ENF_INV_REL_POS_PERIODIC:
      for (int i = 0; i < 2; ++i) {
        float s, c; sincospif(pr[i], &s, &c);
        g[i] = 3.14159265358979323846f *
               (-s * ACC(i, 2 * i) + c * ACC(i, 2 * i + 1) + c * ACC(2 + i, 2 * i) + s * ACC(2 + i, 2 * i + 1));
      }
      break;
    case ENF_INV_PONITA: {
      float o0, o1; sincosf(pr[2], &o1, &o0);
      float a00 = ACC(0, 0), a01 = ACC(0, 1), a02 = ACC(0, 2), a10 = ACC(1, 0), a11 = ACC(1, 1), a12 = ACC(1, 2);
      g[0] = -a02 * o0 + a12 * o1;
      g[1] = -a02 * o1 - a12 * o0;
      float do0 = a00 - a02 * pr[0] + a11 - a12 * pr[1];
      float do1 = a01 - a02 * pr[1] - a10 + a12 * pr[0];
      if (sa) { do0 += ACC(2, 3); do1 += ACC(2, 4); }
      g[2] = -o1 * do0 + o0 * do1;
      if (np) {
        g[0] += 2.f * (pr[0] * ACC(W, 2) - ACC(W, 0));
        g[1] += 2.f * (pr[1] * ACC(W, 2) - ACC(W, 1));
      }
    } break;
    case ENF_INV_POLAR_PERIODIC: {
      float dphi[3], dth[3]; sph_unit_grad(pr[0], pr[1], dphi, dth);
      for (int j = 0; j < 3; ++j) { g[0] += ACC(0, j) * dphi[j]; g[1] += ACC(0, j) * dth[j]; }
    } break;
    case ENF_INV_LATITUDE_PERIODIC: case ENF_INV_BALL_LAT: {
      float s, c; sincosf(pr[0], &s, &c);
      g[1] = ACC(1, 3);
      g[0] = -s * ACC(2, 1) + c * ACC(2, 2) - c * ACC(3, 1) - s * ACC(3, 2);
      if (kind == ENF_INV_BALL_LAT) g[3] = ACC(5, 3);
      if (win_kind == ENF_WIN_SPH) {
        float dphi[3], dth[3]; sph_unit_grad(pr[0], pr[1], dphi, dth);
        for (int j = 0; j < 3; ++j) { g[0] += ACC(W, 4 + j) * dphi[j]; g[1] += ACC(W, 4 + j) * dth[j]; }
      }
    } break;
    case ENF_INV_BALL: {
      float sa, ca, sb, cb, sg, cg;
      sincosf(pr[0], &sa, &ca); sincosf(pr[1], &sb, &cb); sincosf(pr[2], &sg, &cg);
      float R0[3] = {ca * cb, ca * sb * sg - sa * cg, ca * sb * cg + sa * sg};
      float R1[3] = {sa * cb, sa * sb * sg + ca * cg, sa * sb * cg - ca * sg};
      float dB0[3] = {-ca * sb, ca * cb * sg, ca * cb * cg};
      float dB1[3] = {-sa * sb, sa * cb * sg, sa * cb * cg};
      float dB2[3] = {-cb, -sb * sg, -sb * cg};
      float dG0[3] = {0.f, ca * sb * cg + sa * sg, -ca * sb * sg + sa * cg};
      float dG1[3] = {0.f, sa * sb * cg - ca * sg, -sa * sb * sg - ca * cg};
      float dG2[3] = {0.f, cb * cg, -cb * sg};
      for (int j = 0; j < 3; ++j) {
        g[0] += ACC(0, j) * (-R1[j]) + ACC(1, j) * R0[j];                         // dR/dalpha: row0' = -row1, row1' = row0
        g[1] += ACC(0, j) * dB0[j] + ACC(1, j) * dB1[j] + ACC(2, j) * dB2[j];
        g[2] += ACC(0, j) * dG0[j] + ACC(1, j) * dG1[j] + ACC(2, j) * dG2[j];
      }
      g[3] = ACC(4, 4);
      if (win_kind == ENF_WIN_SPH) {
        float dphi[3], dth[3]; sph_unit_grad(pr[0], pr[1], dphi, dth);
        for (int j = 0; j < 3; ++j) { g[0] += ACC(W, j) * dphi[j]; g[1] += ACC(W, j) * dth[j]; }
      }
    } break;
  }
#undef ACC
  for (int i = 0; i < P; ++i) dp[t * P + i] = g[i];
}

// Adjoint of query_features_kernel for one row: g[0..3] = d(row xr) of the record cotangent d[8].  `sa`: the self-attention
// variant (Ponita2D also reads the orientation xr[2]; coordinate rows of the ponita decode are only Dx = 2 wide).
__device__ __forceinline__ void query_features_adjoint(int kind, int Dx, const float* xr, const float* d, float* g, bool sa) {
  switch (kind) {
    case ENF_INV_REL_POS: case ENF_INV_NORM_REL_POS: case ENF_INV_ABS_POS:
      for (int i = 0; i < Dx; ++i) g[i] = d[i];
      break;
    case ENF_INV_REL_POS_PERIODIC:
      for (int i = 0; i < 2; ++i) {
        float s, c; sincospif(xr[i], &s, &c);
        g[i] = 3.14159265358979323846f * (-s * d[2 * i] + c * d[2 * i + 1]);
      }
      break;
    case ENF_INV_PONITA: {
      float s = 0.f, c = 0.f;
      if (sa) sincosf(xr[2], &s, &c);
      g[0] = d[0]; g[1] = d[1];
      if (sa) g[2] = -s * d[3] + c * d[4];
    } break;
    case ENF_INV_POLAR_PERIODIC: {
      float dphi[3], dth[3]; sph_unit_grad(xr[0], xr[1], dphi, dth);
      for (int j = 0; j < 3; ++j) { g[0] += d[j] * dphi[j]; g[1] += d[j] * dth[j]; }
    } break;
    case ENF_INV_LATITUDE_PERIODIC: case ENF_INV_BALL_LAT: {
      float s, c; sincosf(xr[0], &s, &c);
      float dphi[3], dth[3]; sph_unit_grad(xr[0], xr[1], dphi, dth);
      g[1] = d[0];
      g[0] = -s * d[1] + c * d[2];
      for (int j = 0; j < 3; ++j) { g[0] += d[4 + j] * dphi[j]; g[1] += d[4 + j] * dth[j]; }
      if (kind == ENF_INV_BALL_LAT) g[2] = d[7];
    } break;
    case ENF_INV_BALL: {
      float dphi[3], dth[3]; sph_unit_grad(xr[0], xr[1], dphi, dth);
      for (int j = 0; j < 3; ++j) { g[0] += d[j] * dphi[j]; g[1] += d[j] * dth[j]; }
      g[2] = d[3];
    } break;
  }
}

// d(xi record) -> d(raw pose) ACCUMULATED into dp, for poses used as queries (self-attention variant; rows of width P)
__global__ void query_features_bwd_kernel(int kind, int Dx, int P, int64_t total, const float* __restrict__ p,
                                          const float* __restrict__ dxi, float* __restrict__ dp) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  float g[4] = {0.f, 0.f, 0.f, 0.f};
  query_features_adjoint(kind, Dx, p + t * P, dxi + t * ENF_F_XI, g, true);
  for (int i = 0; i < P; ++i) dp[t * P + i] += g[i];
}

// d(xi record) [B,C,8] -> dx, OVERWRITTEN, for the coordinate queries of the decode (sa = 0).  One thread per row of x
// (total = Bx*C rows of width Dx); nsum > 1 (shared grid, Bx = 1): the record cotangents of the nsum fields are summed first
// (the record map is the same for every field, so the sum commutes with its adjoint).
__global__ void coord_features_bwd_kernel(int kind, int Dx, int64_t total, int nsum, int64_t field_stride, const float* __restrict__ x,
                                          const float* __restrict__ dxi, float* __restrict__ dx) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  float d[ENF_F_XI];
#pragma unroll
  for (int f = 0; f < ENF_F_XI; ++f) d[f] = 0.f;
  for (int b = 0; b < nsum; ++b) {
    const float4* src = reinterpret_cast<const float4*>(dxi + b * field_stride + t * ENF_F_XI);
    const float4 u = src[0], v = src[1];
    d[0] += u.x; d[1] += u.y; d[2] += u.z; d[3] += u.w; d[4] += v.x; d[5] += v.y; d[6] += v.z; d[7] += v.w;
  }
  float g[4] = {0.f, 0.f, 0.f, 0.f};
  query_features_adjoint(kind, Dx, x + t * Dx, d, g, false);
  for (int i = 0; i < Dx; ++i) dx[t * Dx + i] = g[i];
}

// ---- elementwise glue of the self-attention blocks (residual adds, the gelu between blocks; nef.py:62-64, 225-226) ------
__global__ void add_kernel(float* __restrict__ out, const float* __restrict__ a, const float* __restrict__ b, int64_t n) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) out[t] = a[t] + b[t];
}
__global__ void add_gelu_kernel(float* __restrict__ pre, float* __restrict__ out, const float* __restrict__ a, const float* __restrict__ b, int64_t n) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) { const float v = a[t] + b[t]; pre[t] = v; out[t] = enf_gelu(v); }
}
__global__ void mul_gelu_grad_kernel(float* __restrict__ out, const float* __restrict__ g, const float* __restrict__ pre, int64_t n) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) out[t] = g[t] * enf_gelu_grad(pre[t]);
}

// ---- LayerNorm rows (flax: eps 1e-6, var = E[x^2]-E[x]^2), optional gelu on the input --------------
__global__ void __launch_bounds__(256) ln_fwd_kernel(const float* __restrict__ in, int64_t M, int N,
                                                     const float* __restrict__ g, const float* __restrict__ b,
                                                     float* __restrict__ out_core, float* __restrict__ out_aff,
                                                     float* __restrict__ rstd_out, int gelu_in, int rnd) {
  const int lane = threadIdx.x & 31;
  int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = warp; r < M; r += nwarps) {
    const float* row = in + r * N;
    float s = 0.f, s2 = 0.f;
    for (int j = lane; j < N; j += 32) {
      float v = row[j];
      if (gelu_in) v = enf_gelu(v);
      s += v; s2 += v * v;
    }
    s = warp_sum(s); s2 = warp_sum(s2);
    float mu = s / N;
    float var = fmaxf(s2 / N - mu * mu, 0.f);
    float rstd = rsqrtf(var + 1e-6f);
    if (lane == 0 && rstd_out) rstd_out[r] = rstd;
    for (int j = lane; j < N; j += 32) {
      float v = row[j];
      if (gelu_in) v = enf_gelu(v);
      float c = (v - mu) * rstd;
      if (out_core) out_core[r * N + j] = c;
      if (out_aff) out_aff[r * N + j] = enf_maybe_round(c * g[j] + b[j], rnd);
    }
  }
}

// dy = cotangent of (core*g + b).  dx = cotangent of the (pre-gelu) input.  dg/db accumulated atomically.
// One warp per row, one pass: a lane keeps its (<= 16) elements of dy / core in registers between the row
// reduction and the write-back (float4 accesses when N % 128 == 0).
__device__ __forceinline__ float gelu_grad_fast(float x) {
  const float c0 = 0.7978845608028654f, c1 = 0.7978845608028654f * 0.044715f;
  float x2 = x * x, t;
  float u = x * fmaf(c1, x2, c0);
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(u));
  float s = fmaf(0.5f, t, 0.5f);
  return fmaf(x * s * fmaf(-2.f, s, 2.f), fmaf(3.f * c1, x2, c0), s);
}
template <int NV4>     // N == 128 * NV4
__global__ void __launch_bounds__(256) ln_bwd_vec_kernel(const float* dy, const float* __restrict__ core,
                                                         const float* __restrict__ rstd, const float* __restrict__ g,
                                                         const float* __restrict__ pre, int64_t M,
                                                         float* dx, float* __restrict__ dg,
                                                         float* __restrict__ db, int gelu_in, int rnd, int fast_gelu) {
  constexpr int N = 128 * NV4;
  const int lane = threadIdx.x & 31;
  int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  float4 gv[NV4], pg[NV4], pb[NV4];
#pragma unroll
  for (int t = 0; t < NV4; ++t) {
    gv[t] = *reinterpret_cast<const float4*>(g + 128 * t + 4 * lane);
    pg[t] = make_float4(0.f, 0.f, 0.f, 0.f); pb[t] = pg[t];
  }
  for (int64_t r = warp; r < M; r += nwarps) {
    float4 d[NV4], c[NV4], p[NV4];
#pragma unroll
    for (int t = 0; t < NV4; ++t) {
      d[t] = *reinterpret_cast<const float4*>(dy + r * N + 128 * t + 4 * lane);
      c[t] = __ldg(reinterpret_cast<const float4*>(core + r * N + 128 * t + 4 * lane));
      if (gelu_in) p[t] = __ldg(reinterpret_cast<const float4*>(pre + r * N + 128 * t + 4 * lane));
    }
    const float rs = rstd[r];
    float m1 = 0.f, m2 = 0.f;
#pragma unroll
    for (int t = 0; t < NV4; ++t) {
      float a0 = d[t].x * gv[t].x, a1 = d[t].y * gv[t].y, a2 = d[t].z * gv[t].z, a3 = d[t].w * gv[t].w;
      m1 += (a0 + a1) + (a2 + a3);
      m2 += (a0 * c[t].x + a1 * c[t].y) + (a2 * c[t].z + a3 * c[t].w);
    }
    m1 = warp_sum(m1) * (1.f / N); m2 = warp_sum(m2) * (1.f / N);
#pragma unroll
    for (int t = 0; t < NV4; ++t) {
      float dv[4] = {d[t].x, d[t].y, d[t].z, d[t].w}, cv[4] = {c[t].x, c[t].y, c[t].z, c[t].w};
      float gg[4] = {gv[t].x, gv[t].y, gv[t].z, gv[t].w}, pv[4] = {0.f, 0.f, 0.f, 0.f}, o[4];
      if (gelu_in) { pv[0] = p[t].x; pv[1] = p[t].y; pv[2] = p[t].z; pv[3] = p[t].w; }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float v = rs * (dv[q] * gg[q] - m1 - cv[q] * m2);
        if (gelu_in) v *= fast_gelu ? gelu_grad_fast(pv[q]) : enf_gelu_grad(pv[q]);
        o[q] = enf_maybe_round(v, rnd);
      }
      *reinterpret_cast<float4*>(dx + r * N + 128 * t + 4 * lane) = make_float4(o[0], o[1], o[2], o[3]);
      pg[t].x += dv[0] * cv[0]; pg[t].y += dv[1] * cv[1]; pg[t].z += dv[2] * cv[2]; pg[t].w += dv[3] * cv[3];
      pb[t].x += dv[0]; pb[t].y += dv[1]; pb[t].z += dv[2]; pb[t].w += dv[3];
    }
  }
  if (dg) {
    // block-level reduction in shared memory first: 8 warps -> one atomic per column per block
    __shared__ float sg[N], sb[N];
    for (int j = threadIdx.x; j < N; j += blockDim.x) { sg[j] = 0.f; sb[j] = 0.f; }
    __syncthreads();
#pragma unroll
    for (int t = 0; t < NV4; ++t) {
      const int j = 128 * t + 4 * lane;
      atomicAdd(&sg[j], pg[t].x); atomicAdd(&sg[j + 1], pg[t].y); atomicAdd(&sg[j + 2], pg[t].z); atomicAdd(&sg[j + 3], pg[t].w);
      atomicAdd(&sb[j], pb[t].x); atomicAdd(&sb[j + 1], pb[t].y); atomicAdd(&sb[j + 2], pb[t].z); atomicAdd(&sb[j + 3], pb[t].w);
    }
    __syncthreads();
    for (int j = threadIdx.x; j < N; j += blockDim.x) { atomicAdd(dg + j, sg[j]); atomicAdd(db + j, sb[j]); }
  }
}

__global__ void __launch_bounds__(256) ln_bwd_kernel(const float* dy, const float* __restrict__ core,
                                                     const float* __restrict__ rstd, const float* __restrict__ g,
                                                     const float* __restrict__ pre, int64_t M, int N,
                                                     float* dx, float* __restrict__ dg,
                                                     float* __restrict__ db, int gelu_in, int rnd) {
  const int lane = threadIdx.x & 31;
  int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  float pg[16], pb[16];      // N <= 512
#pragma unroll
  for (int t = 0; t < 16; ++t) { pg[t] = 0.f; pb[t] = 0.f; }
  for (int64_t r = warp; r < M; r += nwarps) {
    float m1 = 0.f, m2 = 0.f;
    for (int j = lane; j < N; j += 32) {
      float dc = dy[r * N + j] * g[j];
      m1 += dc; m2 += dc * core[r * N + j];
    }
    m1 = warp_sum(m1) / N; m2 = warp_sum(m2) / N;
    float rs = rstd[r];
#pragma unroll
    for (int t = 0; t < 16; ++t) {
      int j = lane + 32 * t;
      if (j < N) {
        float d = dy[r * N + j], c = core[r * N + j];
        float v = rs * (d * g[j] - m1 - c * m2);
        if (gelu_in) v *= enf_gelu_grad(pre[r * N + j]);
        dx[r * N + j] = enf_maybe_round(v, rnd);
        pg[t] += d * c; pb[t] += d;
      }
    }
  }
  if (dg) {
#pragma unroll
    for (int t = 0; t < 16; ++t) {
      int j = lane + 32 * t;
      if (j < N) { atomicAdd(dg + j, pg[t]); atomicAdd(db + j, pb[t]); }
    }
  }
}

// out[n] += sum_m G[m][n] (* mul[m][n])
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ G, int64_t M, int N, int64_t ld,
                                                     float* __restrict__ out, const float* __restrict__ mul,
                                                     int64_t ld_mul, int64_t rows_per_block) {
  int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  int64_t r1 = r0 + rows_per_block; if (r1 > M) r1 = M;
  for (int n = threadIdx.x; n < N; n += blockDim.x) {
    float s = 0.f;
    for (int64_t r = r0; r < r1; ++r) {
      float v = G[r * ld + n];
      if (mul) v *= mul[r * ld_mul + n];
      s += v;
    }
    atomicAdd(out + n, s);
  }
}

__global__ void rowscale_kernel(const float* __restrict__ W, const float* __restrict__ g, float* __restrict__ out,
                                int rows, int cols) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)rows * cols) return;
  out[t] = W[t] * g[t / cols];
}

// out[i][j] = g[i]*A[i][j] + u[i]*v[j]
__global__ void mul_rows_kernel(float* __restrict__ out, const float* __restrict__ A, const float* __restrict__ g,
                                int rows, int cols, const float* __restrict__ u, const float* __restrict__ v) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)rows * cols) return;
  int i = t / cols, j = t % cols;
  float r = g[i] * A[t];
  if (u) r += u[i] * v[j];
  out[t] = r;
}

__global__ void add_outer_kernel(float* __restrict__ C, int64_t ldc, const float* __restrict__ u,
                                 const float* __restrict__ v, int M, int N) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)M * N) return;
  int i = t / N, j = t % N;
  C[i * ldc + j] += u[i] * v[j];
}

// out[i] = sum_j A[i][j]*B[i][j]   (one warp per row)
__global__ void rowdot_kernel(const float* __restrict__ A, const float* __restrict__ Bm, float* __restrict__ out,
                              int rows, int cols) {
  int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows) return;
  float s = 0.f;
  for (int j = lane; j < cols; j += 32) s += A[(int64_t)warp * cols + j] * Bm[(int64_t)warp * cols + j];
  s = warp_sum(s);
  if (lane == 0) out[warp] = s;
}

// ---- FiLM effective weights: Weff[b,z,h] = W2g_gamma[:,h] diag(v0[b,z,h]) + W2g_beta[:,h] -----------
__global__ void __launch_bounds__(256) weff_kernel(int d, int H, const float* __restrict__ W2g,
                                                   const float* __restrict__ b2g, const float* __restrict__ v0,
                                                   float* __restrict__ Weff, float* __restrict__ beff, int rnd) {
  const int64_t bzh = blockIdx.x;
  const int h = bzh % H;
  const int64_t bz = bzh / H;
  const int Hd = H * d;
  const float* v = v0 + bz * Hd + h * d;
  float* out = Weff + bzh * d * d;
  for (int e = threadIdx.x; e < d * d; e += blockDim.x) {
    int i = e / d, j = e % d;
    out[e] = enf_maybe_round(W2g[(int64_t)i * 2 * Hd + h * d + j] * v[j] + W2g[(int64_t)i * 2 * Hd + Hd + h * d + j], rnd);
  }
  for (int j = threadIdx.x; j < d; j += blockDim.x)
    beff[bzh * d + j] = v[j] * (1.f + b2g[h * d + j]) + b2g[Hd + h * d + j];
}

__global__ void __launch_bounds__(128) weff_bwd_dv0_kernel(int d, int H, const float* __restrict__ W2g,
                                                           const float* __restrict__ b2g,
                                                           const float* __restrict__ dWeff,
                                                           const float* __restrict__ dbeff, float* __restrict__ dv0) {
  const int64_t bzh = blockIdx.x;
  const int h = bzh % H;
  const int64_t bz = bzh / H;
  const int Hd = H * d;
  for (int j = threadIdx.x; j < d; j += blockDim.x) {
    float s = dbeff[bzh * d + j] * (1.f + b2g[h * d + j]);
    const float* dw = dWeff + bzh * d * d + j;
    for (int i = 0; i < d; ++i) s += W2g[(int64_t)i * 2 * Hd + h * d + j] * dw[(int64_t)i * d];
    dv0[bz * Hd + h * d + j] = s;
  }
}

// grid (d [i] + 1 [bias row], H, chunks); block d threads [j]
__global__ void __launch_bounds__(128) weff_bwd_dw_kernel(int d, int H, int64_t BZ, int64_t per_chunk,
                                                          const float* __restrict__ v0,
                                                          const float* __restrict__ dWeff,
                                                          const float* __restrict__ dbeff,
                                                          float* __restrict__ dW2g, float* __restrict__ db2g) {
  const int i = blockIdx.x, h = blockIdx.y;
  const int Hd = H * d;
  int64_t z0 = (int64_t)blockIdx.z * per_chunk, z1 = z0 + per_chunk;
  if (z1 > BZ) z1 = BZ;
  for (int j = threadIdx.x; j < d; j += blockDim.x) {
    float sg = 0.f, sb = 0.f;
    for (int64_t bz = z0; bz < z1; ++bz) {
      float v = v0[bz * Hd + h * d + j];
      float g = (i < d) ? dWeff[(bz * H + h) * d * d + (int64_t)i * d + j] : dbeff[(bz * H + h) * d + j];
      sg += g * v; sb += g;
    }
    if (i < d) {
      atomicAdd(dW2g + (int64_t)i * 2 * Hd + h * d + j, sg);
      atomicAdd(dW2g + (int64_t)i * 2 * Hd + Hd + h * d + j, sb);
    } else {
      atomicAdd(db2g + h * d + j, sg);
      atomicAdd(db2g + Hd + h * d + j, sb);
    }
  }
}

__global__ void transpose_kernel(const float* __restrict__ in, float* __restrict__ out, int rows, int cols) {
  __shared__ float tile[32][33];
  const float* src = in + (int64_t)blockIdx.z * rows * cols;
  float* dst = out + (int64_t)blockIdx.z * rows * cols;
  int c = blockIdx.x * 32 + threadIdx.x;
  for (int k = threadIdx.y; k < 32; k += blockDim.y) {
    int r = blockIdx.y * 32 + k;
    if (r < rows && c < cols) tile[k][threadIdx.x] = src[(int64_t)r * cols + c];
  }
  __syncthreads();
  int r2 = blockIdx.y * 32 + threadIdx.x;
  for (int k = threadIdx.y; k < 32; k += blockDim.y) {
    int c2 = blockIdx.x * 32 + k;
    if (c2 < cols && r2 < rows) dst[(int64_t)c2 * rows + r2] = tile[threadIdx.x][k];
  }
}

inline int blocks_for(int64_t n, int per) { return (int)((n + per - 1) / per); }

}  // namespace

int enf_launch_rowscale(cudaStream_t st, const float* W, const float* g, float* out, int rows, int cols) {
  rowscale_kernel<<<blocks_for((int64_t)rows * cols, 256), 256, 0, st>>>(W, g, out, rows, cols);
  return 1;
}

// ---- the decode MLP's last layer (d -> O, O <= 4): three memory-bound "thin" products -------------------------------------
namespace {
// out[m,o] = sum_k act(A[m,k]) W[k,o] + b[o]; one warp per row, float4 lanes over k
template <int O>
__global__ void __launch_bounds__(256) thin_out_kernel(const float* __restrict__ A, const float* __restrict__ W, const float* __restrict__ b,
                                                       float* __restrict__ out, int64_t M, int d, int act_a, int out_bf16) {
  const int lane = threadIdx.x & 31;
  int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t m = warp; m < M; m += nwarps) {
    float acc[O];
#pragma unroll
    for (int o = 0; o < O; ++o) acc[o] = 0.f;
    for (int k = 4 * lane; k < d; k += 128) {
      const float4 a4 = __ldg(reinterpret_cast<const float4*>(A + m * d + k));
      float a[4] = {a4.x, a4.y, a4.z, a4.w};
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        if (act_a) a[t] = enf_gelu(a[t]);
#pragma unroll
        for (int o = 0; o < O; ++o) acc[o] = fmaf(a[t], __ldg(W + (k + t) * O + o), acc[o]);
      }
    }
#pragma unroll
    for (int o = 0; o < O; ++o) acc[o] = warp_sum(acc[o]);
    if (lane == 0) {
#pragma unroll
      for (int o = 0; o < O; ++o) {
        if (out_bf16) reinterpret_cast<__nv_bfloat16*>(out)[m * O + o] = __float2bfloat16_rn(acc[o] + b[o]);
        else out[m * O + o] = acc[o] + b[o];
      }
    }
  }
}
// dX[m,k] = (sum_o dO[m,o] W[k,o]) gelu'(pre[m,k]); one thread per 4 consecutive k
template <int O>
__global__ void __launch_bounds__(256) thin_dgrad_kernel(const float* __restrict__ dO, const float* __restrict__ W,
                                                         const float* __restrict__ pre, float* __restrict__ dX, int64_t M, int d) {
  const int64_t total = M * (d / 4);
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t m = t / (d / 4);
    const int k = (int)(t % (d / 4)) * 4;
    float g[O];
#pragma unroll
    for (int o = 0; o < O; ++o) g[o] = __ldg(dO + m * O + o);
    const float4 p4 = __ldg(reinterpret_cast<const float4*>(pre + m * d + k));
    const float p[4] = {p4.x, p4.y, p4.z, p4.w};
    float r[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      float s = 0.f;
#pragma unroll
      for (int o = 0; o < O; ++o) s = fmaf(g[o], __ldg(W + (k + q) * O + o), s);
      r[q] = s * enf_gelu_grad(p[q]);
    }
    *reinterpret_cast<float4*>(dX + m * d + k) = make_float4(r[0], r[1], r[2], r[3]);
  }
}
// dW[k,o] += sum_m act(A[m,k]) dO[m,o] ; db[o] += sum_m dO[m,o]; thread = column k, rows_per_block rows per block
template <int O>
__global__ void __launch_bounds__(256) thin_wgrad_kernel(const float* __restrict__ A, const float* __restrict__ dO, float* __restrict__ dW,
                                                         float* __restrict__ db, int64_t M, int d, int act_a, int64_t rows_per_block) {
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  int64_t r1 = r0 + rows_per_block; if (r1 > M) r1 = M;
  for (int k = threadIdx.x; k < d; k += blockDim.x) {
    float acc[O], bs[O];
#pragma unroll
    for (int o = 0; o < O; ++o) { acc[o] = 0.f; bs[o] = 0.f; }
#pragma unroll 4
    for (int64_t m = r0; m < r1; ++m) {
      float a = __ldg(A + m * d + k);
      if (act_a) a = enf_gelu(a);
#pragma unroll
      for (int o = 0; o < O; ++o) { const float g = __ldg(dO + m * O + o); acc[o] = fmaf(a, g, acc[o]); bs[o] += g; }
    }
#pragma unroll
    for (int o = 0; o < O; ++o) {
      atomicAdd(dW + (int64_t)k * O + o, acc[o]);
      if (k == 0 && db) atomicAdd(db + o, bs[o]);
    }
  }
}
}  // namespace

bool enf_thin_supported(int d, int O) { return O >= 1 && O <= 4 && d % 4 == 0; }
int enf_launch_thin_out(cudaStream_t st, const float* A, const float* W, const float* b, float* out, int64_t M, int d, int O, int act_a,
                        int out_bf16) {
  int blocks = (int)((M + 7) / 8); if (blocks > 148 * 16) blocks = 148 * 16;
  switch (O) {
    case 1: thin_out_kernel<1><<<blocks, 256, 0, st>>>(A, W, b, out, M, d, act_a, out_bf16); break;
    case 2: thin_out_kernel<2><<<blocks, 256, 0, st>>>(A, W, b, out, M, d, act_a, out_bf16); break;
    case 3: thin_out_kernel<3><<<blocks, 256, 0, st>>>(A, W, b, out, M, d, act_a, out_bf16); break;
    case 4: thin_out_kernel<4><<<blocks, 256, 0, st>>>(A, W, b, out, M, d, act_a, out_bf16); break;
    default: return -1;
  }
  return 1;
}
int enf_launch_thin_dgrad(cudaStream_t st, const float* dO, const float* W, const float* pre, float* dX, int64_t M, int d, int O) {
  int64_t total = M * (d / 4);
  int blocks = (int)((total + 255) / 256); if (blocks > 148 * 16) blocks = 148 * 16;
  switch (O) {
    case 1: thin_dgrad_kernel<1><<<blocks, 256, 0, st>>>(dO, W, pre, dX, M, d); break;
    case 2: thin_dgrad_kernel<2><<<blocks, 256, 0, st>>>(dO, W, pre, dX, M, d); break;
    case 3: thin_dgrad_kernel<3><<<blocks, 256, 0, st>>>(dO, W, pre, dX, M, d); break;
    case 4: thin_dgrad_kernel<4><<<blocks, 256, 0, st>>>(dO, W, pre, dX, M, d); break;
    default: return -1;
  }
  return 1;
}
int enf_launch_thin_wgrad(cudaStream_t st, const float* A, const float* dO, float* dW, float* db, int64_t M, int d, int O, int act_a) {
  int64_t rpb = (M + 148 * 8 - 1) / (148 * 8);
  if (rpb < 16) rpb = 16;
  int blocks = (int)((M + rpb - 1) / rpb);
  int threads = d < 256 ? ((d + 31) / 32) * 32 : 256;
  switch (O) {
    case 1: thin_wgrad_kernel<1><<<blocks, threads, 0, st>>>(A, dO, dW, db, M, d, act_a, rpb); break;
    case 2: thin_wgrad_kernel<2><<<blocks, threads, 0, st>>>(A, dO, dW, db, M, d, act_a, rpb); break;
    case 3: thin_wgrad_kernel<3><<<blocks, threads, 0, st>>>(A, dO, dW, db, M, d, act_a, rpb); break;
    case 4: thin_wgrad_kernel<4><<<blocks, threads, 0, st>>>(A, dO, dW, db, M, d, act_a, rpb); break;
    default: return -1;
  }
  return 1;
}

int enf_launch_colsum(cudaStream_t st, const float* G, int64_t M, int N, int64_t ld, float* out, const float* mul,
                      int64_t ld_mul) {
  if (M <= 0) return 0;
  int64_t rpb = (M + 591) / 592;
  if (rpb < 8) rpb = 8;
  int blocks = (int)((M + rpb - 1) / rpb);
  colsum_kernel<<<blocks, 256, 0, st>>>(G, M, N, ld, out, mul, ld_mul, rpb);
  return 1;
}

int enf_launch_ln_fwd(cudaStream_t st, const float* in, int64_t M, int N, const float* g, const float* b,
                      float* out_core, float* out_affine, float* rstd, int gelu_in, int round_affine) {
  int blocks = (int)((M + 7) / 8); if (blocks > 148 * 16) blocks = 148 * 16;
  ln_fwd_kernel<<<blocks, 256, 0, st>>>(in, M, N, g, b, out_core, out_affine, rstd, gelu_in, round_affine);
  return 1;
}

int enf_launch_ln_bwd(cudaStream_t st, const float* dy, const float* core, const float* rstd, const float* g,
                      const float* pre, int64_t M, int N, float* dx, float* dg, float* db, int gelu_in, int round_dx, int fast_gelu) {
  int blocks = (int)((M + 7) / 8); if (blocks > 148 * 8) blocks = 148 * 8;
  // fast_gelu: tanh.approx in gelu' (tensor-core precision mode only: the result feeds tf32 operands anyway)
  if (N == 128) ln_bwd_vec_kernel<1><<<blocks, 256, 0, st>>>(dy, core, rstd, g, pre, M, dx, dg, db, gelu_in, round_dx, fast_gelu);
  else if (N == 256) ln_bwd_vec_kernel<2><<<blocks, 256, 0, st>>>(dy, core, rstd, g, pre, M, dx, dg, db, gelu_in, round_dx, fast_gelu);
  else if (N == 384) ln_bwd_vec_kernel<3><<<blocks, 256, 0, st>>>(dy, core, rstd, g, pre, M, dx, dg, db, gelu_in, round_dx, fast_gelu);
  else if (N == 512) ln_bwd_vec_kernel<4><<<blocks, 256, 0, st>>>(dy, core, rstd, g, pre, M, dx, dg, db, gelu_in, round_dx, fast_gelu);
  else ln_bwd_kernel<<<blocks, 256, 0, st>>>(dy, core, rstd, g, pre, M, N, dx, dg, db, gelu_in, round_dx);
  return 1;
}

int enf_launch_add(cudaStream_t st, float* out, const float* a, const float* b, int64_t n) {
  add_kernel<<<blocks_for(n, 256), 256, 0, st>>>(out, a, b, n);
  return 1;
}
int enf_launch_add_gelu(cudaStream_t st, float* pre, float* out, const float* a, const float* b, int64_t n) {
  add_gelu_kernel<<<blocks_for(n, 256), 256, 0, st>>>(pre, out, a, b, n);
  return 1;
}
int enf_launch_mul_gelu_grad(cudaStream_t st, float* out, const float* g, const float* pre, int64_t n) {
  mul_gelu_grad_kernel<<<blocks_for(n, 256), 256, 0, st>>>(out, g, pre, n);
  return 1;
}

int enf_launch_query_features(cudaStream_t st, const EnfDesc& d, const float* x, int64_t xbs, int Bx, float* xi) {
  int64_t total = (int64_t)Bx * d.C;
  query_features_kernel<<<blocks_for(total, 256), 256, 0, st>>>(d.invariant_kind, d.Dx, d.C, total, x, xbs, xi, d.Dx, 0);
  return 1;
}

// the "queries" are the latent poses themselves (latent ODE model, ponita_ode_g.py:154 `self.invariant(p, p)`): rows of raw
// poses [total][P] -> xi records; self-attention variant of the invariant
int enf_launch_pose_features(cudaStream_t st, int kind, int Dx, int P, int64_t total, const float* p, float* xi) {
  query_features_kernel<<<blocks_for(total, 256), 256, 0, st>>>(kind, Dx, 1, total, p, (int64_t)P, xi, P, 1);
  return 1;
}
int enf_launch_pose_features_bwd(cudaStream_t st, int kind, int Dx, int P, int64_t total, const float* p, const float* dxi, float* dp) {
  query_features_bwd_kernel<<<blocks_for(total, 128), 128, 0, st>>>(kind, Dx, P, total, p, dxi, dp);
  return 1;
}
int enf_launch_coord_features_bwd(cudaStream_t st, const EnfDesc& d, const float* x, int Bx, const float* dxi, float* dx) {
  const int64_t total = (int64_t)Bx * d.C;
  coord_features_bwd_kernel<<<blocks_for(total, 128), 128, 0, st>>>(d.invariant_kind, d.Dx, total, Bx == 1 ? d.B : 1,
                                                                     (int64_t)d.C * ENF_F_XI, x, dxi, dx);
  return 1;
}
int enf_launch_pose_record(cudaStream_t st, int kind, int Dx, int P, int I, int64_t total, const float* p, float* lam) {
  latent_record_kernel<<<blocks_for(total, 128), 128, 0, st>>>(kind, Dx, P, I, total, p, lam, 1);
  return 1;
}
int enf_launch_pose_record_bwd(cudaStream_t st, int kind, int Dx, int P, int I, int win_kind, int64_t total, const float* p, const float* dlam, float* dp) {
  latent_record_bwd_kernel<<<blocks_for(total, 128), 128, 0, st>>>(kind, Dx, P, I, win_kind, total, p, dlam, dp, 1);
  return 1;
}

int enf_launch_latent_record(cudaStream_t st, const EnfDesc& d, const float* p, float* lam) {
  EnfInvariantLayout r = enf_record_layout(d.invariant_kind, d.Dx, d.use_window);
  int64_t total = (int64_t)d.B * d.Z;
  latent_record_kernel<<<blocks_for(total, 128), 128, 0, st>>>(d.invariant_kind, d.Dx, r.P, r.I, total, p, lam, 0);
  return 1;
}

int enf_launch_latent_record_bwd(cudaStream_t st, const EnfDesc& d, const float* p, const float* dlam, float* dp) {
  EnfInvariantLayout r = enf_record_layout(d.invariant_kind, d.Dx, d.use_window);
  int64_t total = (int64_t)d.B * d.Z;
  latent_record_bwd_kernel<<<blocks_for(total, 128), 128, 0, st>>>(d.invariant_kind, d.Dx, r.P, r.I, r.win_kind, total,
                                                                   p, dlam, dp, 0);
  return 1;
}

int enf_launch_weff(cudaStream_t st, const EnfDesc& d, const float* W2g, const float* b2g, const float* v0,
                    float* Weff, float* beff, int round_weff) {
  int64_t bzh = (int64_t)d.B * d.Z * d.H;
  weff_kernel<<<(unsigned)bzh, 256, 0, st>>>(d.d, d.H, W2g, b2g, v0, Weff, beff, round_weff);
  return 1;
}

int enf_launch_weff_bwd(cudaStream_t st, const EnfDesc& d, const float* W2g, const float* b2g, const float* v0,
                        const float* dWeff, const float* dbeff, float* dW2g, float* db2g, float* dv0) {
  int64_t BZ = (int64_t)d.B * d.Z;
  weff_bwd_dv0_kernel<<<(unsigned)(BZ * d.H), 128, 0, st>>>(d.d, d.H, W2g, b2g, dWeff, dbeff, dv0);
  int chunks = (int)((BZ + 63) / 64); if (chunks > 64) chunks = 64;
  int64_t per = (BZ + chunks - 1) / chunks;
  chunks = (int)((BZ + per - 1) / per);
  weff_bwd_dw_kernel<<<dim3(d.d + 1, d.H, chunks), 128, 0, st>>>(d.d, d.H, BZ, per, v0, dWeff, dbeff, dW2g, db2g);
  return 2;
}

namespace {
__global__ void split_lo_kernel(EnfSplitList l) {
  const int k = blockIdx.y;
  if (k >= l.count) return;
  const float* src = l.src[k];
  float* dst = l.dst[k];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < l.n[k]; i += gridDim.x * blockDim.x) {
    float v = src[i];
    dst[i] = v - __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
  }
}
}  // namespace
int enf_launch_split_lo(cudaStream_t st, const EnfSplitList& l) {
  if (l.count <= 0) return 0;
  split_lo_kernel<<<dim3(64, l.count), 256, 0, st>>>(l);
  return 1;
}
int enf_launch_add_outer(cudaStream_t st, float* C, int64_t ldc, const float* u, const float* v, int M, int N) {
  add_outer_kernel<<<blocks_for((int64_t)M * N, 256), 256, 0, st>>>(C, ldc, u, v, M, N);
  return 1;
}

int enf_launch_rowdot(cudaStream_t st, const float* A, const float* Bm, float* out, int rows, int cols) {
  rowdot_kernel<<<blocks_for((int64_t)rows * 32, 256), 256, 0, st>>>(A, Bm, out, rows, cols);
  return 1;
}

int enf_launch_mul_rows(cudaStream_t st, float* out, const float* A, const float* g, int rows, int cols,
                        const float* u, const float* v) {
  mul_rows_kernel<<<blocks_for((int64_t)rows * cols, 256), 256, 0, st>>>(out, A, g, rows, cols, u, v);
  return 1;
}

int enf_launch_transpose(cudaStream_t st, const float* in, float* out, int rows, int cols, int batch) {
  dim3 grid((cols + 31) / 32, (rows + 31) / 32, batch);
  transpose_kernel<<<grid, dim3(32, 8), 0, st>>>(in, out, rows, cols);
  return 1;
}
