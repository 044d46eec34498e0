// Latent ODE model (PonitaODEGen, experiments/fitting/ode_models/ponita_ode_g.py:90-257) and its fixed-step solver
// (trainer_utils/solvers.py:73-162) behind the C ABI of include/enf_ode_b200.h.  fp32 throughout (the reference computes
// this model in float32; it is ~0.3 % of the FLOPs of the ENF decode it sits next to).
//
// Data layout: a "pair row" is (b, r, s) = receiver latent r (the `x` argument of invariant(p, p)), sender latent s (the `p`
// argument), n = B*Z*Z rows; a "latent row" is (b, z), m = B*Z rows.  The invariants are evaluated from the same per-pose
// records the ENF kernels use (xi for the receiver, Lam for the sender: enf_stages.cu), so every invariant kind and its
// Jacobian exist once.  Dense layers over pair / latent rows run on the library's strided fp32 GEMM (enf_gemm.cu); the
// kernels here are what is specific to the model: tensor-power features, the separable group convolution
// ('bsc,brsc->brc'), the vector read-out over relative positions / orientations, and their backward passes.
#include <string>
#include <string.h>

#include "enf_common.cuh"
#include "../../include/enf_ode_b200.h"

int enf_set_error(int code, const char* msg);     // enf_api.cu (thread-local message behind enf_last_error)

namespace {

struct Dims {
  int B, Z, L, Hd, Bd, NL, W, deg, Dx, kind;
  EnfInvariantLayout rec;                            // of the pair invariants (rec.I: their width, rec.P: the pose width)
  int npos, nori, S, F, Fp;                         // Fp: row stride of the feature matrices (F rounded up to 32)
  int64_t m, n;
};

int validate(const EnfOdeDesc* D, Dims* o) {
  if (!D) return enf_set_error(ENF_ERR_NULL_POINTER, "desc is NULL");
  if (D->B <= 0 || D->Z <= 0 || D->L <= 0 || D->hidden <= 0 || D->basis <= 0 || D->widen <= 0)
    return enf_set_error(ENF_ERR_BAD_DESC, "B, Z, L, hidden, basis, widen must be positive");
  if (D->layers < 1 || D->layers > ENF_ODE_MAX_LAYERS) return enf_set_error(ENF_ERR_UNSUPPORTED, "layers must be 1..ENF_ODE_MAX_LAYERS");
  if (D->degree < 0 || D->degree > 5) return enf_set_error(ENF_ERR_UNSUPPORTED, "degree must be 0..5");
  for (int i = 0; i < 6; ++i) if (D->reserved[i]) return enf_set_error(ENF_ERR_BAD_DESC, "reserved fields must be 0");
  EnfInvariantLayout r = enf_record_layout(D->invariant_kind, D->Dx, 0);
  if (r.I < 0) return enf_set_error(ENF_ERR_BAD_DESC, "unknown invariant_kind");
  const int k = D->invariant_kind;
  const bool dx_ok = (k == ENF_INV_REL_POS || k == ENF_INV_NORM_REL_POS || k == ENF_INV_ABS_POS) ? (D->Dx >= 1 && D->Dx <= 3)
                   : (k == ENF_INV_BALL || k == ENF_INV_BALL_LAT) ? D->Dx == 3 : D->Dx == 2;
  if (!dx_ok) return enf_set_error(ENF_ERR_BAD_DESC, "num_in (Dx) does not match the invariant");
  Dims d;
  d.B = D->B; d.Z = D->Z; d.L = D->L; d.Hd = D->hidden; d.Bd = D->basis; d.NL = D->layers; d.W = D->widen * D->hidden;
  d.deg = D->degree; d.Dx = D->Dx; d.kind = k;
  d.rec = r;
  if (k == ENF_INV_PONITA) d.rec.I = 3;           // Ponita2D (get_sa_invariant), ponita.py:46-86
  d.nori = k == ENF_INV_PONITA ? 1 : 0; d.npos = d.rec.P - d.nori;
  d.S = d.L + d.nori;
  int64_t F = 0, pw = 1;
  for (int t = 0; t <= d.deg; ++t) { pw *= d.rec.I; F += pw; }
  if (F > 4096) return enf_set_error(ENF_ERR_UNSUPPORTED, "tensor-power feature width above 4096");
  d.F = (int)F;
  d.Fp = (d.F + 31) / 32 * 32;
  d.m = (int64_t)d.B * d.Z; d.n = d.m * d.Z;
  if (d.n * (int64_t)(d.F > d.Hd ? d.F : d.Hd) > ((int64_t)1 << 40)) return enf_set_error(ENF_ERR_UNSUPPORTED, "B*Z*Z too large for one call");
  if (d.Z > 65535) return enf_set_error(ENF_ERR_UNSUPPORTED, "Z must be <= 65535");
  *o = d;
  return ENF_OK;
}

// ---- workspace ----------------------------------------------------------------------------------------------------------
struct Ws {
  int64_t total = 0;
  int64_t take(int64_t n) { int64_t o = total; total += (n + 63) / 64 * 64; return o; }
  // forward state
  int64_t lam, xi, inv, poly, h0p, h0, kbp, kb, am1, hin[ENF_ODE_MAX_LAYERS + 1];
  int64_t K[ENF_ODE_MAX_LAYERS], cv[ENF_ODE_MAX_LAYERS], core[ENF_ODE_MAX_LAYERS], ln[ENF_ODE_MAX_LAYERS], rstd[ENF_ODE_MAX_LAYERS],
      l1p[ENF_ODE_MAX_LAYERS], l1a[ENF_ODE_MAX_LAYERS];
  int64_t scalar, hs, wpair, ptab;
  int64_t w0p, w0lo, w1lo, cklo[ENF_ODE_MAX_LAYERS];      // zero-padded kb_w0 (Fp rows) and the low parts W - trunc_tf32(W) for the 3-term tf32 products
  // backward scratch
  int64_t g_scalar, g_ha, g_hb, g_l1, g_ln, g_c, g_K, g_kb, g_kbp, g_h0, g_poly, g_inv, gw, g_lam, g_xi, ssum, gpe, rosum;
  // solver scratch
  int64_t kp[4], ka[4], tp, ta, sp, sa;
};

Ws make_ws(const Dims& d) {
  Ws w;
  w.lam = w.take(d.m * ENF_LAM_SIZE); w.xi = w.take(d.m * ENF_F_XI);
  w.inv = w.take(d.n * d.rec.I); w.poly = w.take(d.n * d.Fp);
  w.h0p = w.take(d.n * d.Hd); w.h0 = w.take(d.n * d.Hd); w.kbp = w.take(d.n * d.Bd); w.kb = w.take(d.n * d.Bd);
  w.am1 = w.take(d.m * d.L);
  for (int l = 0; l <= d.NL; ++l) w.hin[l] = w.take(d.m * d.Hd);
  for (int l = 0; l < d.NL; ++l) {
    w.K[l] = w.take(d.n * d.Hd); w.cv[l] = w.take(d.m * d.Hd); w.core[l] = w.take(d.m * d.Hd); w.ln[l] = w.take(d.m * d.Hd);
    w.rstd[l] = w.take(d.m); w.l1p[l] = w.take(d.m * d.W); w.l1a[l] = w.take(d.m * d.W);
  }
  w.scalar = w.take(d.m * d.S); w.hs = w.take(d.m * 2); w.wpair = w.take(d.n * 2); w.ptab = w.take(d.Fp);
  w.w0p = w.take((int64_t)d.Fp * d.Hd); w.w0lo = w.take((int64_t)d.Fp * d.Hd); w.w1lo = w.take((int64_t)d.Hd * d.Bd);
  for (int l = 0; l < d.NL; ++l) w.cklo[l] = w.take((int64_t)d.Bd * d.Hd);
  w.g_scalar = w.take(d.m * d.S); w.g_ha = w.take(d.m * d.Hd); w.g_hb = w.take(d.m * d.Hd); w.g_l1 = w.take(d.m * d.W);
  w.g_ln = w.take(d.m * d.Hd); w.g_c = w.take(d.m * d.Hd); w.g_K = w.take(d.n * d.Hd); w.g_kb = w.take(d.n * d.Bd);
  w.g_kbp = w.take(d.n * d.Bd); w.g_h0 = w.take(d.n * d.Hd); w.g_poly = w.take(d.n * d.Fp); w.g_inv = w.take(d.n * d.rec.I);
  w.gw = w.take(d.n * 2); w.g_lam = w.take(d.m * ENF_LAM_SIZE); w.g_xi = w.take(d.m * ENF_F_XI); w.ssum = w.take(d.m * 2);
  w.gpe = w.take(d.m * 8); w.rosum = w.take(2 * (d.rec.I + d.Hd));
  for (int i = 0; i < 4; ++i) { w.kp[i] = w.take(d.m * d.rec.P); w.ka[i] = w.take(d.m * d.L); }
  w.tp = w.take(d.m * d.rec.P); w.ta = w.take(d.m * d.L); w.sp = w.take(d.m * d.rec.P); w.sa = w.take(d.m * d.L);
  return w;
}

inline int nblocks(int64_t n, int per) { return (int)((n + per - 1) / per); }

// ---- kernels ------------------------------------------------------------------------------------------------------------
__global__ void ode_am1_kernel(const float* __restrict__ a, float* __restrict__ am1, int64_t total) {      // ponita_ode_g.py:233
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < total) am1[t] = a[t] - 1.f;
}

// kb_w0 [F][Hd] -> zero-padded copy [Fp][Hd] (the tensor-core GEMMs take whole 32-feature blocks)
__global__ void ode_pad_rows_kernel(const float* __restrict__ src, float* __restrict__ dst, int64_t n_src, int64_t n_dst) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n_dst) dst[t] = t < n_src ? src[t] : 0.f;
}

// Digit table of the tensor-power features (PolynomialFeatures, ponita_ode_g.py:22-27): feature e of level k (k + 1 factors) is
// prod_t u[digit_t(e)]; entry = k | digit_0 << 4 | digit_1 << 8 | ... (digits < 8).  Built once per call: the pair kernels then
// decode a word with shifts instead of dividing by the runtime invariant width per feature.
__global__ void ode_poly_table_kernel(int I, int F, uint32_t* __restrict__ tab) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= F) return;
  int idx = e, size = I, k = 0;
  while (idx >= size) { idx -= size; size *= I; ++k; }
  uint32_t w = (uint32_t)k;
  for (int t = 0; t <= k; ++t) { w |= (uint32_t)(idx % I) << (4 + 4 * t); idx /= I; }
  tab[e] = w;
}

// invariants of every pair row and their tensor powers [u, u (x) u, ...].  One warp per pair row; lanes stride over the F
// features (coalesced stores).
__global__ void __launch_bounds__(256) ode_inv_poly_kernel(EnfRecordLayout rl, int F, int Fp, int Z, int64_t n,
                                                           const float* __restrict__ lam, const float* __restrict__ xi,
                                                           const uint32_t* __restrict__ tab, float* __restrict__ inv,
                                                           float* __restrict__ poly) {
  __shared__ float su[8][8];
  const int lane = threadIdx.x & 31, wl = threadIdx.x >> 5;
  const int64_t row = (int64_t)blockIdx.x * 8 + wl;
  if (row >= n) return;
  const int64_t br = row / Z;                    // (b, r)
  const int64_t bs = (br / Z) * Z + row % Z;     // (b, s)
  if (lane < rl.I) {
    float u = record_row(rl, lam + bs * ENF_LAM_SIZE, xi + br * ENF_F_XI, lane);
    su[wl][lane] = u;
    inv[row * rl.I + lane] = u;
  }
  __syncwarp();
  const float* u = su[wl];
  for (int e = lane; e < Fp; e += 32) {
    float prod = 0.f;                              // columns F .. Fp - 1: zero padding (the row stride is a multiple of 32)
    if (e < F) {
      const uint32_t w = __ldg(tab + e);
      const int k = w & 15;
      prod = u[(w >> 4) & 7];
      if (k > 0) prod *= u[(w >> 8) & 7];
      if (k > 1) prod *= u[(w >> 12) & 7];
      if (k > 2) prod *= u[(w >> 16) & 7];
      if (k > 3) prod *= u[(w >> 20) & 7];
      if (k > 4) prod *= u[(w >> 24) & 7];
    }
    poly[row * Fp + e] = prod;
  }
}

// g_inv[row][i] += sum_e g_poly[row][e] d(poly_e)/d(u_i): per feature, the product of the other factors (prefix x suffix) goes
// to the digit's slot of a per-warp shared accumulator (shared atomics: at most 6 distinct addresses per warp)
__global__ void __launch_bounds__(256) ode_poly_bwd_kernel(int I, int F, int Fp, int64_t n, const float* __restrict__ inv,
                                                           const float* __restrict__ g_poly, const uint32_t* __restrict__ tab,
                                                           float* __restrict__ g_inv) {
  __shared__ float su[8][8];
  const int lane = threadIdx.x & 31, wl = threadIdx.x >> 5;
  const int64_t row = (int64_t)blockIdx.x * 8 + wl;
  if (row >= n) return;
  if (lane < 8) su[wl][lane] = lane < I ? inv[row * I + lane] : 0.f;
  __syncwarp();
  const float* u = su[wl];
  float acc[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int e = lane; e < F; e += 32) {
    const uint32_t w = __ldg(tab + e);
    const int k = w & 15;
    const float g = g_poly[row * Fp + e];
    int dg[6]; float f[6];
#pragma unroll
    for (int t = 0; t < 6; ++t) { dg[t] = (w >> (4 + 4 * t)) & 7; f[t] = t <= k ? u[dg[t]] : 1.f; }
    // suffix products: suf[t] = prod_{t' > t} f[t']
    float suf[6];
    suf[5] = 1.f;
#pragma unroll
    for (int t = 4; t >= 0; --t) suf[t] = suf[t + 1] * f[t + 1];
    float pre = g;
#pragma unroll
    for (int t = 0; t < 6; ++t) {
      if (t <= k) {
        const float part = pre * suf[t];
#pragma unroll
        for (int i = 0; i < 6; ++i) acc[i] += dg[t] == i ? part : 0.f;
      }
      pre *= f[t];
    }
  }
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    const float v = warp_sum(acc[i]);
    if (lane == 0 && i < I) g_inv[row * I + i] += v;
  }
}

// SepGconv (ponita_ode_g.py:81-86): c[b,r,ch] = sum_s h[b,s,ch] K[b,r,s,ch] + bias[ch]
__global__ void ode_conv_fwd_kernel(int Z, int Hd, int64_t total, const float* __restrict__ h, const float* __restrict__ K,
                                    const float* __restrict__ bias, float* __restrict__ c) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const int ch = (int)(t % Hd);
  const int64_t br = t / Hd, b = br / Z;
  const float* hp = h + b * Z * Hd + ch;
  const float* kp = K + br * Z * Hd + ch;
  float s = 0.f;
  for (int z = 0; z < Z; ++z) s = fmaf(hp[(int64_t)z * Hd], kp[(int64_t)z * Hd], s);
  c[t] = s + bias[ch];
}
// g_K[b,r,s,ch] = g_c[b,r,ch] h[b,s,ch]
__global__ void ode_conv_bwd_k_kernel(int Z, int Hd, int64_t total, const float* __restrict__ g_c, const float* __restrict__ h,
                                      float* __restrict__ g_K) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const int ch = (int)(t % Hd);
  const int64_t row = t / Hd, br = row / Z, bs = (br / Z) * Z + row % Z;
  g_K[t] = g_c[br * Hd + ch] * h[bs * Hd + ch];
}
// g_h[b,s,ch] = sum_r g_c[b,r,ch] K[b,r,s,ch]
__global__ void ode_conv_bwd_h_kernel(int Z, int Hd, int64_t total, const float* __restrict__ g_c, const float* __restrict__ K,
                                      float* __restrict__ g_h) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const int ch = (int)(t % Hd);
  const int64_t bs = t / Hd, b = bs / Z, s = bs % Z;
  float acc = 0.f;
  for (int r = 0; r < Z; ++r) acc = fmaf(g_c[(b * Z + r) * Hd + ch], K[((b * Z + r) * Z + s) * Hd + ch], acc);
  g_h[t] = acc;
}

// hs[b,s,0/1] = h[b,s,:] . ro_rel[I:] / ro_ori[I:]   (the sender-feature part of the vector read-outs, ponita_ode_g.py:177-189)
__global__ void __launch_bounds__(256) ode_hs_kernel(int I, int Hd, int64_t m, const float* __restrict__ h, const float* __restrict__ ro_rel,
                                                     const float* __restrict__ ro_ori, float* __restrict__ hs) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= m) return;
  float a = 0.f, o = 0.f;
  for (int c = lane; c < Hd; c += 32) {
    const float v = h[row * Hd + c];
    a = fmaf(v, ro_rel[I + c], a);
    if (ro_ori) o = fmaf(v, ro_ori[I + c], o);
  }
  a = warp_sum(a); o = warp_sum(o);
  if (lane == 0) { hs[row * 2] = a; hs[row * 2 + 1] = o; }
}

// vector read-out + assembly of (dp/dt, da/dt) (ponita_ode_g.py:170-190, 236-244).  One warp per receiver (b, r).
__global__ void __launch_bounds__(256) ode_readout_fwd_kernel(int I, int Z, int P, int npos, int nori, int L, int S, int64_t m,
                                                              const float* __restrict__ p, const float* __restrict__ inv,
                                                              const float* __restrict__ hs, const float* __restrict__ scalar,
                                                              const float* __restrict__ ro_rel, const float* __restrict__ ro_ori,
                                                              float* __restrict__ wpair, float* __restrict__ dp_dt, float* __restrict__ da_dt) {
  const int lane = threadIdx.x & 31;
  const int64_t br = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (br >= m) return;
  const int64_t b = br / Z;
  float pr[4] = {0.f, 0.f, 0.f, 0.f}, vec[4] = {0.f, 0.f, 0.f, 0.f};
  for (int k = 0; k < npos; ++k) pr[k] = p[br * P + k];
  for (int s = lane; s < Z; s += 32) {
    const int64_t bs = b * Z + s, row = br * Z + s;
    float wr = hs[bs * 2], wo = hs[bs * 2 + 1];
    for (int i = 0; i < I; ++i) {
      const float u = inv[row * I + i];
      wr = fmaf(u, ro_rel[i], wr);
      if (nori) wo = fmaf(u, ro_ori[i], wo);
    }
    wpair[row * 2] = wr; wpair[row * 2 + 1] = wo;
    for (int k = 0; k < npos; ++k) vec[k] = fmaf(wr, pr[k] - p[bs * P + k], vec[k]);
    if (nori) {
      float so, co; sincosf(p[bs * P + npos], &so, &co);
      vec[0] = fmaf(wo, co, vec[0]); vec[1] = fmaf(wo, so, vec[1]);
    }
  }
  const float invz = 1.f / (float)Z;
  for (int k = 0; k < npos; ++k) { const float v = warp_sum(vec[k]); if (lane == 0) dp_dt[br * P + k] = v * invz; }
  if (nori && lane == 0) dp_dt[br * P + npos] = scalar[br * S + L];
  for (int j = lane; j < L; j += 32) da_dt[br * L + j] = scalar[br * S + j];
}

// backward of the read-out, receiver side: cotangents of the pair weights (gw), of the invariants (g_inv =), of the receiver's
// position (gpe[.,0..3] =), read-out weight gradients of the invariant rows (rosum[0..I), rosum[I+Hd..I+Hd+I)) and g_scalar
__global__ void __launch_bounds__(256) ode_readout_bwd_r_kernel(int I, int Hd, int Z, int P, int npos, int nori, int L, int S, int64_t m,
                                                                const float* __restrict__ p, const float* __restrict__ inv,
                                                                const float* __restrict__ wpair, const float* __restrict__ g_dp,
                                                                const float* __restrict__ g_da, const float* __restrict__ ro_rel,
                                                                const float* __restrict__ ro_ori, float* __restrict__ gw,
                                                                float* __restrict__ g_inv, float* __restrict__ gpe,
                                                                float* __restrict__ rosum, float* __restrict__ g_scalar) {
  const int lane = threadIdx.x & 31;
  const int64_t br = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (br >= m) return;
  const int64_t b = br / Z;
  const float invz = 1.f / (float)Z;
  float pr[4] = {0.f, 0.f, 0.f, 0.f}, gv[4] = {0.f, 0.f, 0.f, 0.f};
  for (int k = 0; k < npos; ++k) { pr[k] = p[br * P + k]; gv[k] = g_dp[br * P + k] * invz; }
  float swr = 0.f, dro_r[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, dro_o[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int s = lane; s < Z; s += 32) {
    const int64_t bs = b * Z + s, row = br * Z + s;
    float gwr = 0.f, gwo = 0.f;
    for (int k = 0; k < npos; ++k) gwr = fmaf(gv[k], pr[k] - p[bs * P + k], gwr);
    if (nori) {
      float so, co; sincosf(p[bs * P + npos], &so, &co);
      gwo = gv[0] * co + gv[1] * so;
    }
    gw[row * 2] = gwr; gw[row * 2 + 1] = gwo;
    swr += wpair[row * 2];
#pragma unroll
    for (int i = 0; i < 6; ++i) if (i < I) {
      const float u = inv[row * I + i];
      g_inv[row * I + i] = gwr * ro_rel[i] + (nori ? gwo * ro_ori[i] : 0.f);
      dro_r[i] = fmaf(gwr, u, dro_r[i]); dro_o[i] = fmaf(gwo, u, dro_o[i]);
    }
  }
  swr = warp_sum(swr);
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    const float a = warp_sum(dro_r[i]), o = warp_sum(dro_o[i]);
    if (lane == 0 && i < I && rosum) { atomicAdd(rosum + i, a); if (nori) atomicAdd(rosum + I + Hd + i, o); }
  }
  if (lane == 0) {
    for (int k = 0; k < 4; ++k) gpe[br * 8 + k] = k < npos ? swr * gv[k] : 0.f;
    if (nori) g_scalar[br * S + L] = g_dp[br * P + npos];
  }
  for (int j = lane; j < L; j += 32) g_scalar[br * S + j] = g_da[br * L + j];
}
// sender side: sums over receivers -> ssum (cotangent of hs), position / orientation cotangents of the sender (gpe +=)
__global__ void __launch_bounds__(256) ode_readout_bwd_s_kernel(int Z, int P, int npos, int nori, int64_t m, const float* __restrict__ p,
                                                                const float* __restrict__ wpair, const float* __restrict__ gw,
                                                                const float* __restrict__ g_dp, float* __restrict__ ssum,
                                                                float* __restrict__ gpe) {
  const int lane = threadIdx.x & 31;
  const int64_t bs = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (bs >= m) return;
  const int64_t b = bs / Z, s = bs % Z;
  const float invz = 1.f / (float)Z;
  float sr = 0.f, so = 0.f, gp[4] = {0.f, 0.f, 0.f, 0.f}, go[2] = {0.f, 0.f};
  for (int r = lane; r < Z; r += 32) {
    const int64_t br = b * Z + r, row = br * Z + s;
    sr += gw[row * 2]; so += gw[row * 2 + 1];
    const float wr = wpair[row * 2] * invz, wo = wpair[row * 2 + 1] * invz;
    for (int k = 0; k < npos; ++k) gp[k] = fmaf(-wr, g_dp[br * P + k], gp[k]);
    if (nori) { go[0] = fmaf(wo, g_dp[br * P], go[0]); go[1] = fmaf(wo, g_dp[br * P + 1], go[1]); }
  }
  sr = warp_sum(sr); so = warp_sum(so);
  for (int k = 0; k < 4; ++k) gp[k] = warp_sum(gp[k]);
  go[0] = warp_sum(go[0]); go[1] = warp_sum(go[1]);
  if (lane == 0) {
    ssum[bs * 2] = sr; ssum[bs * 2 + 1] = so;
    for (int k = 0; k < npos; ++k) gpe[bs * 8 + k] += gp[k];
    float ga = 0.f;
    if (nori) { float sn, cs; sincosf(p[bs * P + npos], &sn, &cs); ga = -sn * go[0] + cs * go[1]; }
    gpe[bs * 8 + 4] = ga;
  }
}
// g_h[bs,c] += ssum[bs,0] ro_rel[I+c] + ssum[bs,1] ro_ori[I+c];  rosum[I+c] += sum_bs ssum[bs,0] h[bs,c] (block partial sums)
__global__ void ode_readout_bwd_h_kernel(int I, int Hd, int64_t m, const float* __restrict__ ssum, const float* __restrict__ h,
                                         const float* __restrict__ ro_rel, const float* __restrict__ ro_ori, float* __restrict__ g_h,
                                         float* __restrict__ rosum) {
  const int c = blockIdx.y * blockDim.x + threadIdx.x;
  if (c >= Hd) return;
  const int64_t rows_per = (m + gridDim.x - 1) / gridDim.x, r0 = blockIdx.x * rows_per, r1 = r0 + rows_per < m ? r0 + rows_per : m;
  const float wr = ro_rel[I + c], wo = ro_ori ? ro_ori[I + c] : 0.f;
  float ar = 0.f, ao = 0.f;
  for (int64_t bs = r0; bs < r1; ++bs) {
    const float sr = ssum[bs * 2], so = ssum[bs * 2 + 1], hv = h[bs * Hd + c];
    g_h[bs * Hd + c] += sr * wr + so * wo;
    ar = fmaf(sr, hv, ar); ao = fmaf(so, hv, ao);
  }
  if (rosum) { atomicAdd(rosum + I + c, ar); if (ro_ori) atomicAdd(rosum + I + Hd + I + c, ao); }
}

// g_lam[bs][i][f] = sum_r dq[(b,r,s)][i] xi[(b,r)][f]   (what the ENF pair backward accumulates per latent, enf_stages.cu)
__global__ void ode_inv_bwd_lam_kernel(EnfRecordLayout rl, int Z, int64_t total, const float* __restrict__ inv,
                                       const float* __restrict__ g_inv, const float* __restrict__ xi, float* __restrict__ g_lam) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const int f = (int)(t % ENF_F_XI), i = (int)((t / ENF_F_XI) % ENF_R_LAM);
  const int64_t bs = t / ENF_LAM_SIZE, b = bs / Z, s = bs % Z;
  float acc = 0.f;
  if (i < rl.I)
    for (int r = 0; r < Z; ++r) {
      const int64_t br = b * Z + r, row = br * Z + s;
      const float du = g_inv[row * rl.I + i];
      acc = fmaf(rl.row_kind == ENF_ROW_SQDIST_SQRT ? record_sqrt_adjoint(du, inv[row * rl.I + i]) : du, xi[br * ENF_F_XI + f], acc);
    }
  g_lam[t] = acc;
}
// g_xi[br][f] = sum_s sum_i du Lam[(b,s)][i][f]  (DOT rows)  |  sum_s -2 dq (Lam[(b,s)][0][f] - xi[br][f])  (SQDIST rows, f < nsq)
__global__ void ode_inv_bwd_xi_kernel(EnfRecordLayout rl, int Z, int64_t total, const float* __restrict__ inv,
                                      const float* __restrict__ g_inv, const float* __restrict__ lam, const float* __restrict__ xi,
                                      float* __restrict__ g_xi) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const int f = (int)(t % ENF_F_XI);
  const int64_t br = t / ENF_F_XI, b = br / Z;
  float acc = 0.f;
  if (rl.row_kind == ENF_ROW_DOT) {
    for (int s = 0; s < Z; ++s) {
      const int64_t row = br * Z + s;
      const float* Lm = lam + (b * Z + s) * ENF_LAM_SIZE + f;
      for (int i = 0; i < rl.I; ++i) acc = fmaf(g_inv[row * rl.I + i], Lm[i * ENF_F_XI], acc);
    }
  } else if (f < rl.nsq) {
    const float x = xi[br * ENF_F_XI + f];
    for (int s = 0; s < Z; ++s) {
      const int64_t row = br * Z + s;
      const float du = g_inv[row * rl.I];
      const float dq = rl.row_kind == ENF_ROW_SQDIST_SQRT ? record_sqrt_adjoint(du, inv[row * rl.I]) : du;
      acc = fmaf(-2.f * dq, lam[(b * Z + s) * ENF_LAM_SIZE + f] - x, acc);
    }
  }
  g_xi[t] = acc;
}
// gp[bz][:] += gpe: positions (first npos), orientation angle (slot 4)
__global__ void ode_add_gpe_kernel(int P, int npos, int nori, int64_t m, const float* __restrict__ gpe, float* __restrict__ gp) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= m) return;
  for (int k = 0; k < npos; ++k) gp[t * P + k] += gpe[t * 8 + k];
  if (nori) gp[t * P + npos] += gpe[t * 8 + 4];
}
// scatter the read-out weight sums into the caller's leaves
__global__ void ode_ro_scatter_kernel(int n, const float* __restrict__ rosum, float* __restrict__ d_rel, float* __restrict__ d_ori) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  d_rel[t] = rosum[t];
  if (d_ori) d_ori[t] = rosum[n + t];
}
// out = g * gelu'(pre)   (cotangent through the second gelu of the kernel-basis MLP)
__global__ void ode_mul_gelu_grad_kernel(int64_t total, const float* __restrict__ g, const float* __restrict__ pre, float* __restrict__ out) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < total) out[t] = g[t] * enf_gelu_grad(pre[t]);
}
// y = x + c0 k0 (+ c1 k1 + c2 k2 + c3 k3)   (tree-mapped solver updates, solvers.py:85-107)
__global__ void ode_axpy_kernel(int64_t total, const float* __restrict__ x, float c0, const float* __restrict__ k0, float c1,
                                const float* __restrict__ k1, float c2, const float* __restrict__ k2, float c3, const float* __restrict__ k3,
                                float* __restrict__ y) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  float v = c0 * k0[t];
  if (k1) v += c1 * k1[t];
  if (k2) v += c2 * k2[t];
  if (k3) v += c3 * k3[t];
  y[t] = x[t] + v;
}
// trajectories are [B, T+1, Z, .]: copy state rows [B, Z, w] into time slot `step`
__global__ void ode_store_traj_kernel(int Z, int w, int T1, int step, int64_t total, const float* __restrict__ x, float* __restrict__ traj) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const int64_t per = (int64_t)Z * w, b = t / per, rem = t % per;
  traj[(b * T1 + step) * per + rem] = x[t];
}

struct Run {
  cudaStream_t st;
  float* ws;
  bool failed = false;
  int launches = 0;
  void gemm(int64_t M, int N, int K, EnfMat A, EnfMat B, EnfMat C, const EnfGemmOpts& o = EnfGemmOpts()) {
    if (M <= 0 || N <= 0) return;
    int r = enf_gemm(st, (int)M, N, K, A, B, C, o);
    if (r < 0) failed = true; else launches += r;
  }
};
EnfGemmOpts o_bias(const float* b, float* gelu_out = nullptr) { EnfGemmOpts o; o.bias = b; o.gelu_out = gelu_out; return o; }
// 3-term tf32 tensor-core product when the shape allows (b_lo: the weight's low part, laid out like the weight)
EnfGemmOpts o_tc(EnfGemmOpts o, const float* b_lo) { o.tc = 1; o.b_lo = b_lo; return o; }
EnfGemmOpts o_acc() { EnfGemmOpts o; o.accumulate = 1; return o; }
EnfGemmOpts o_dgelu(const float* pre) { EnfGemmOpts o; o.mul_gelu_grad = pre; return o; }

int check_ptrs(const Dims& d, const EnfOdeWeights* w, const void* workspace) {
  if (!w) return enf_set_error(ENF_ERR_NULL_POINTER, "weights are NULL");
  if (!w->kb_w0 || !w->kb_b0 || !w->kb_w1 || !w->kb_b1 || !w->stem_w || !w->ro_scalar || !w->ro_rel || (d.nori && !w->ro_ori))
    return enf_set_error(ENF_ERR_NULL_POINTER, "a weight leaf is NULL");
  for (int l = 0; l < d.NL; ++l) {
    const EnfOdeLayer& y = w->layer[l];
    if (!y.conv_k || !y.conv_b || !y.ln_g || !y.ln_b || !y.l1_w || !y.l1_b || !y.l2_w || !y.l2_b)
      return enf_set_error(ENF_ERR_NULL_POINTER, "a ConvBlock weight leaf is NULL");
  }
  if (!workspace || ((uintptr_t)workspace & 255)) return enf_set_error(ENF_ERR_WORKSPACE, "workspace is NULL or not 256-byte aligned");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return enf_set_error(ENF_ERR_NO_DEVICE, "no CUDA device");
  return ENF_OK;
}

int forward(const Dims& d, const Ws& Y, const EnfOdeWeights& w, const float* p, const float* a, float* dp_dt, float* da_dt, Run& R) {
  cudaStream_t st = R.st;
  float* W = R.ws;
  R.launches += enf_launch_pose_record(st, d.kind, d.Dx, d.rec.P, d.rec.I, d.m, p, W + Y.lam);
  R.launches += enf_launch_pose_features(st, d.kind, d.Dx, d.rec.P, d.m, p, W + Y.xi);
  uint32_t* ptab = reinterpret_cast<uint32_t*>(W + Y.ptab);
  ode_poly_table_kernel<<<nblocks(d.F, 128), 128, 0, st>>>(d.rec.I, d.F, ptab);
  ode_inv_poly_kernel<<<nblocks(d.n, 8), 256, 0, st>>>(d.rec, d.F, d.Fp, d.Z, d.n, W + Y.lam, W + Y.xi, ptab, W + Y.inv, W + Y.poly);
  // The pair-row Dense layers run on the tf32 tensor-core kernels as 3-term split products (fp32-level accuracy,
  // enf_gemm_tc.cu) when the shapes allow (hidden, basis multiples of 32, >= 128 pair rows), else on the fp32 kernel: the
  // low parts W - trunc_tf32(W) of the weights they multiply by, and kb_w0 zero-padded to whole 32-feature blocks
  ode_pad_rows_kernel<<<nblocks((int64_t)d.Fp * d.Hd, 256), 256, 0, st>>>(w.kb_w0, W + Y.w0p, (int64_t)d.F * d.Hd, (int64_t)d.Fp * d.Hd);
  {
    EnfSplitList sl;
    int c = 0;
    auto add = [&](const float* src, float* dst, int64_t n) {
      sl.src[c] = src; sl.dst[c] = dst; sl.n[c] = (int)n; ++c;
      if (c == 8) { sl.count = c; R.launches += enf_launch_split_lo(st, sl); c = 0; }
    };
    add(W + Y.w0p, W + Y.w0lo, (int64_t)d.Fp * d.Hd);
    add(w.kb_w1, W + Y.w1lo, (int64_t)d.Hd * d.Bd);
    for (int l = 0; l < d.NL; ++l) add(w.layer[l].conv_k, W + Y.cklo[l], (int64_t)d.Bd * d.Hd);
    if (c) { sl.count = c; R.launches += enf_launch_split_lo(st, sl); }
  }
  // kernel basis: Dense -> gelu -> Dense -> gelu (ponita_ode_g.py:107-109)
  R.gemm(d.n, d.Hd, d.Fp, enf_mat(W + Y.poly, d.Fp), enf_mat(W + Y.w0p, d.Hd), enf_mat(W + Y.h0p, d.Hd), o_tc(o_bias(w.kb_b0, W + Y.h0), W + Y.w0lo));
  R.gemm(d.n, d.Bd, d.Hd, enf_mat(W + Y.h0, d.Hd), enf_mat(w.kb_w1, d.Bd), enf_mat(W + Y.kbp, d.Bd), o_tc(o_bias(w.kb_b1, W + Y.kb), W + Y.w1lo));
  ode_am1_kernel<<<nblocks(d.m * d.L, 256), 256, 0, st>>>(a, W + Y.am1, d.m * d.L);
  R.gemm(d.m, d.Hd, d.L, enf_mat(W + Y.am1, d.L), enf_mat(w.stem_w, d.Hd), enf_mat(W + Y.hin[0], d.Hd));
  for (int l = 0; l < d.NL; ++l) {
    const EnfOdeLayer& y = w.layer[l];
    R.gemm(d.n, d.Hd, d.Bd, enf_mat(W + Y.kb, d.Bd), enf_mat(y.conv_k, d.Hd), enf_mat(W + Y.K[l], d.Hd), o_tc(EnfGemmOpts(), W + Y.cklo[l]));
    ode_conv_fwd_kernel<<<nblocks(d.m * d.Hd, 256), 256, 0, st>>>(d.Z, d.Hd, d.m * d.Hd, W + Y.hin[l], W + Y.K[l], y.conv_b, W + Y.cv[l]);
    R.launches += enf_launch_ln_fwd(st, W + Y.cv[l], d.m, d.Hd, y.ln_g, y.ln_b, W + Y.core[l], W + Y.ln[l], W + Y.rstd[l], 0);
    R.gemm(d.m, d.W, d.Hd, enf_mat(W + Y.ln[l], d.Hd), enf_mat(y.l1_w, d.W), enf_mat(W + Y.l1p[l], d.W), o_bias(y.l1_b, W + Y.l1a[l]));
    R.gemm(d.m, d.Hd, d.W, enf_mat(W + Y.l1a[l], d.W), enf_mat(y.l2_w, d.Hd), enf_mat(W + Y.hin[l + 1], d.Hd), o_bias(y.l2_b));
  }
  const float* h = W + Y.hin[d.NL];
  R.gemm(d.m, d.S, d.Hd, enf_mat(h, d.Hd), enf_mat(w.ro_scalar, d.S), enf_mat(W + Y.scalar, d.S));
  ode_hs_kernel<<<nblocks(d.m, 8), 256, 0, st>>>(d.rec.I, d.Hd, d.m, h, w.ro_rel, d.nori ? w.ro_ori : nullptr, W + Y.hs);
  ode_readout_fwd_kernel<<<nblocks(d.m, 8), 256, 0, st>>>(d.rec.I, d.Z, d.rec.P, d.npos, d.nori, d.L, d.S, d.m, p, W + Y.inv, W + Y.hs,
                                                           W + Y.scalar, w.ro_rel, d.nori ? w.ro_ori : nullptr, W + Y.wpair, dp_dt, da_dt);
  R.launches += 6 + 1 * d.NL;
  if (R.failed) return enf_set_error(ENF_ERR_CUDA, "a stage GEMM of the latent ODE model could not be configured");
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return enf_set_error(ENF_ERR_CUDA, (std::string("CUDA error while enqueueing enf_ode_fwd: ") + cudaGetErrorString(e)).c_str());
  return ENF_OK;
}

}  // namespace

extern "C" {

size_t enf_ode_workspace_bytes(const EnfOdeDesc* desc) {
  Dims d;
  if (validate(desc, &d) != ENF_OK) return 0;
  return (size_t)make_ws(d).total * sizeof(float);
}

int enf_ode_fwd(const EnfOdeDesc* desc, const EnfOdeWeights* w, const float* p, const float* a, float* dp_dt, float* da_dt,
                void* workspace, size_t workspace_bytes, enf_stream_t stream) {
  Dims d;
  int rc = validate(desc, &d);
  if (rc != ENF_OK) return rc;
  if (!p || !a || !dp_dt || !da_dt) return enf_set_error(ENF_ERR_NULL_POINTER, "NULL argument");
  if ((rc = check_ptrs(d, w, workspace)) != ENF_OK) return rc;
  Ws Y = make_ws(d);
  if (workspace_bytes < (size_t)Y.total * sizeof(float)) return enf_set_error(ENF_ERR_WORKSPACE, "workspace too small: see enf_ode_workspace_bytes");
  Run R; R.st = (cudaStream_t)stream; R.ws = (float*)workspace;
  return forward(d, Y, *w, p, a, dp_dt, da_dt, R);
}

int enf_ode_bwd(const EnfOdeDesc* desc, const EnfOdeWeights* w, const float* p, const float* a, const float* g_dp, const float* g_da,
                const EnfOdeWeightGrads* dW, float* gp, float* ga, void* workspace, size_t workspace_bytes, enf_stream_t stream) {
  Dims d;
  int rc = validate(desc, &d);
  if (rc != ENF_OK) return rc;
  if (!p || !a || !g_dp || !g_da || !gp || !ga) return enf_set_error(ENF_ERR_NULL_POINTER, "NULL argument");
  if ((rc = check_ptrs(d, w, workspace)) != ENF_OK) return rc;
  Ws Y = make_ws(d);
  if (workspace_bytes < (size_t)Y.total * sizeof(float)) return enf_set_error(ENF_ERR_WORKSPACE, "workspace too small");
  Run R; R.st = (cudaStream_t)stream; R.ws = (float*)workspace;
  cudaStream_t st = R.st;
  float* W = R.ws;
  const bool wg = dW != nullptr;
  auto zero = [&](float* ptr, int64_t n) { if (ptr) cudaMemsetAsync(ptr, 0, n * sizeof(float), st); };
  if (wg) {
    if (!dW->kb_w0 || !dW->kb_b0 || !dW->kb_w1 || !dW->kb_b1 || !dW->stem_w || !dW->ro_scalar || !dW->ro_rel || (d.nori && !dW->ro_ori))
      return enf_set_error(ENF_ERR_NULL_POINTER, "a weight-gradient leaf is NULL");
    zero(dW->kb_w0, (int64_t)d.F * d.Hd); zero(dW->kb_b0, d.Hd); zero(dW->kb_w1, (int64_t)d.Hd * d.Bd); zero(dW->kb_b1, d.Bd);
    zero(dW->stem_w, (int64_t)d.L * d.Hd); zero(dW->ro_scalar, (int64_t)d.Hd * d.S);
    for (int l = 0; l < d.NL; ++l) {
      const EnfOdeLayerGrads& g = dW->layer[l];
      if (!g.conv_k || !g.conv_b || !g.ln_g || !g.ln_b || !g.l1_w || !g.l1_b || !g.l2_w || !g.l2_b)
        return enf_set_error(ENF_ERR_NULL_POINTER, "a ConvBlock weight-gradient leaf is NULL");
      zero(g.conv_k, (int64_t)d.Bd * d.Hd); zero(g.conv_b, d.Hd); zero(g.ln_g, d.Hd); zero(g.ln_b, d.Hd);
      zero(g.l1_w, (int64_t)d.Hd * d.W); zero(g.l1_b, d.W); zero(g.l2_w, (int64_t)d.W * d.Hd); zero(g.l2_b, d.Hd);
    }
    zero(W + Y.rosum, 2 * (d.rec.I + d.Hd));
  }
  const float* ro_ori = d.nori ? w->ro_ori : nullptr;
  float* rosum = wg ? W + Y.rosum : nullptr;
  const float* h = W + Y.hin[d.NL];
  // ---- read-outs ------------------------------------------------------------------------------------------------------------
  ode_readout_bwd_r_kernel<<<nblocks(d.m, 8), 256, 0, st>>>(d.rec.I, d.Hd, d.Z, d.rec.P, d.npos, d.nori, d.L, d.S, d.m, p, W + Y.inv, W + Y.wpair,
                                                             g_dp, g_da, w->ro_rel, ro_ori, W + Y.gw, W + Y.g_inv, W + Y.gpe, rosum,
                                                             W + Y.g_scalar);
  ode_readout_bwd_s_kernel<<<nblocks(d.m, 8), 256, 0, st>>>(d.Z, d.rec.P, d.npos, d.nori, d.m, p, W + Y.wpair, W + Y.gw, g_dp, W + Y.ssum, W + Y.gpe);
  float* g_h = W + Y.g_ha;
  float* g_h2 = W + Y.g_hb;
  R.gemm(d.m, d.Hd, d.S, enf_mat(W + Y.g_scalar, d.S), enf_mat(w->ro_scalar, 1, d.S), enf_mat(g_h, d.Hd));
  if (wg) R.gemm(d.Hd, d.S, (int)d.m, enf_mat(h, 1, d.Hd), enf_mat(W + Y.g_scalar, d.S), enf_mat(dW->ro_scalar, d.S), o_acc());
  {
    int gx = (int)((d.m + 63) / 64); if (gx > 592) gx = 592;
    dim3 grid(gx, (d.Hd + 127) / 128);
    ode_readout_bwd_h_kernel<<<grid, 128, 0, st>>>(d.rec.I, d.Hd, d.m, W + Y.ssum, h, w->ro_rel, ro_ori, g_h, rosum);
  }
  if (wg) ode_ro_scatter_kernel<<<nblocks(d.rec.I + d.Hd, 128), 128, 0, st>>>(d.rec.I + d.Hd, W + Y.rosum, dW->ro_rel, d.nori ? dW->ro_ori : nullptr);
  // ---- interaction layers, last to first; g_kb accumulates the kernel-basis cotangent over the layers -------------------------
  for (int l = d.NL - 1; l >= 0; --l) {
    const EnfOdeLayer& y = w->layer[l];
    // linear_2
    if (wg) {
      R.gemm(d.W, d.Hd, (int)d.m, enf_mat(W + Y.l1a[l], 1, d.W), enf_mat(g_h, d.Hd), enf_mat(dW->layer[l].l2_w, d.Hd), o_acc());
      R.launches += enf_launch_colsum(st, g_h, d.m, d.Hd, d.Hd, dW->layer[l].l2_b, nullptr, 0);
    }
    R.gemm(d.m, d.W, d.Hd, enf_mat(g_h, d.Hd), enf_mat(y.l2_w, 1, d.Hd), enf_mat(W + Y.g_l1, d.W), o_dgelu(W + Y.l1p[l]));
    // linear_1
    if (wg) {
      R.gemm(d.Hd, d.W, (int)d.m, enf_mat(W + Y.ln[l], 1, d.Hd), enf_mat(W + Y.g_l1, d.W), enf_mat(dW->layer[l].l1_w, d.W), o_acc());
      R.launches += enf_launch_colsum(st, W + Y.g_l1, d.m, d.W, d.W, dW->layer[l].l1_b, nullptr, 0);
    }
    R.gemm(d.m, d.Hd, d.W, enf_mat(W + Y.g_l1, d.W), enf_mat(y.l1_w, 1, d.W), enf_mat(W + Y.g_ln, d.Hd));
    // LayerNorm
    R.launches += enf_launch_ln_bwd(st, W + Y.g_ln, W + Y.core[l], W + Y.rstd[l], y.ln_g, nullptr, d.m, d.Hd, W + Y.g_c,
                                    wg ? dW->layer[l].ln_g : nullptr, wg ? dW->layer[l].ln_b : nullptr, 0);
    // SepGconv
    if (wg) R.launches += enf_launch_colsum(st, W + Y.g_c, d.m, d.Hd, d.Hd, dW->layer[l].conv_b, nullptr, 0);
    ode_conv_bwd_k_kernel<<<nblocks(d.n * d.Hd, 256), 256, 0, st>>>(d.Z, d.Hd, d.n * d.Hd, W + Y.g_c, W + Y.hin[l], W + Y.g_K);
    ode_conv_bwd_h_kernel<<<nblocks(d.m * d.Hd, 256), 256, 0, st>>>(d.Z, d.Hd, d.m * d.Hd, W + Y.g_c, W + Y.K[l], g_h2);
    if (wg) R.gemm(d.Bd, d.Hd, (int)d.n, enf_mat(W + Y.kb, 1, d.Bd), enf_mat(W + Y.g_K, d.Hd), enf_mat(dW->layer[l].conv_k, d.Hd), o_acc());
    if (l == d.NL - 1)      // the first contribution overwrites (tensor-core product), the others accumulate
      R.gemm(d.n, d.Bd, d.Hd, enf_mat(W + Y.g_K, d.Hd), enf_mat(y.conv_k, 1, d.Hd), enf_mat(W + Y.g_kb, d.Bd), o_tc(EnfGemmOpts(), W + Y.cklo[l]));
    else {                  // into g_kbp (free until the kernel-basis stage), then added: keeps the product on the tensor-core kernel
      R.gemm(d.n, d.Bd, d.Hd, enf_mat(W + Y.g_K, d.Hd), enf_mat(y.conv_k, 1, d.Hd), enf_mat(W + Y.g_kbp, d.Bd), o_tc(EnfGemmOpts(), W + Y.cklo[l]));
      R.launches += enf_launch_add(st, W + Y.g_kb, W + Y.g_kb, W + Y.g_kbp, d.n * d.Bd);
    }
    float* t = g_h; g_h = g_h2; g_h2 = t;
    R.launches += 2;
  }
  // ---- a_stem ---------------------------------------------------------------------------------------------------------------
  if (wg) R.gemm(d.L, d.Hd, (int)d.m, enf_mat(W + Y.am1, 1, d.L), enf_mat(g_h, d.Hd), enf_mat(dW->stem_w, d.Hd), o_acc());
  R.gemm(d.m, d.L, d.Hd, enf_mat(g_h, d.Hd), enf_mat(w->stem_w, 1, d.Hd), enf_mat(ga, d.L));
  // ---- kernel basis -----------------------------------------------------------------------------------------------------------
  ode_mul_gelu_grad_kernel<<<nblocks(d.n * d.Bd, 256), 256, 0, st>>>(d.n * d.Bd, W + Y.g_kb, W + Y.kbp, W + Y.g_kbp);
  R.launches += 1;
  if (wg) {
    R.gemm(d.Hd, d.Bd, (int)d.n, enf_mat(W + Y.h0, 1, d.Hd), enf_mat(W + Y.g_kbp, d.Bd), enf_mat(dW->kb_w1, d.Bd), o_acc());
    R.launches += enf_launch_colsum(st, W + Y.g_kbp, d.n, d.Bd, d.Bd, dW->kb_b1, nullptr, 0);
  }
  R.gemm(d.n, d.Hd, d.Bd, enf_mat(W + Y.g_kbp, d.Bd), enf_mat(w->kb_w1, 1, d.Bd), enf_mat(W + Y.g_h0, d.Hd), o_tc(o_dgelu(W + Y.h0p), W + Y.w1lo));
  if (wg) {
    R.gemm(d.F, d.Hd, (int)d.n, enf_mat(W + Y.poly, 1, d.Fp), enf_mat(W + Y.g_h0, d.Hd), enf_mat(dW->kb_w0, d.Hd), o_acc());
    R.launches += enf_launch_colsum(st, W + Y.g_h0, d.n, d.Hd, d.Hd, dW->kb_b0, nullptr, 0);
  }
  // cotangent of the features, in column blocks of <= 256 (the tensor-core kernel's widest tile); padded columns come out 0
  for (int c0 = 0; c0 < d.Fp; c0 += 256) {
    const int nc = d.Fp - c0 < 256 ? d.Fp - c0 : 256;
    R.gemm(d.n, nc, d.Hd, enf_mat(W + Y.g_h0, d.Hd), enf_mat(W + Y.w0p + (int64_t)c0 * d.Hd, 1, d.Hd), enf_mat(W + Y.g_poly + c0, d.Fp),
           o_tc(EnfGemmOpts(), W + Y.w0lo + (int64_t)c0 * d.Hd));
  }
  ode_poly_bwd_kernel<<<nblocks(d.n, 8), 256, 0, st>>>(d.rec.I, d.F, d.Fp, d.n, W + Y.inv, W + Y.g_poly, reinterpret_cast<const uint32_t*>(W + Y.ptab), W + Y.g_inv);
  // ---- invariants -> poses (sender side through Lam, receiver side through xi), read-out position terms ------------------------
  ode_inv_bwd_lam_kernel<<<nblocks(d.m * ENF_LAM_SIZE, 256), 256, 0, st>>>(d.rec, d.Z, d.m * ENF_LAM_SIZE, W + Y.inv, W + Y.g_inv,
                                                                           W + Y.xi, W + Y.g_lam);
  ode_inv_bwd_xi_kernel<<<nblocks(d.m * ENF_F_XI, 256), 256, 0, st>>>(d.rec, d.Z, d.m * ENF_F_XI, W + Y.inv, W + Y.g_inv,
                                                                      W + Y.lam, W + Y.xi, W + Y.g_xi);
  R.launches += enf_launch_pose_record_bwd(st, d.kind, d.Dx, d.rec.P, d.rec.I, ENF_WIN_NONE, d.m, p, W + Y.g_lam, gp);
  R.launches += enf_launch_pose_features_bwd(st, d.kind, d.Dx, d.rec.P, d.m, p, W + Y.g_xi, gp);
  ode_add_gpe_kernel<<<nblocks(d.m, 256), 256, 0, st>>>(d.rec.P, d.npos, d.nori, d.m, W + Y.gpe, gp);
  R.launches += 8;
  if (R.failed) return enf_set_error(ENF_ERR_CUDA, "a stage GEMM of the latent ODE backward could not be configured");
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return enf_set_error(ENF_ERR_CUDA, (std::string("CUDA error while enqueueing enf_ode_bwd: ") + cudaGetErrorString(e)).c_str());
  return ENF_OK;
}

int enf_ode_solve(const EnfOdeDesc* desc, const EnfOdeWeights* w, const float* p0, const float* a0, int32_t num_steps, float h,
                  int32_t method, float* p_traj, float* a_traj, void* workspace, size_t workspace_bytes, enf_stream_t stream) {
  Dims d;
  int rc = validate(desc, &d);
  if (rc != ENF_OK) return rc;
  if (!p0 || !a0 || !p_traj || !a_traj) return enf_set_error(ENF_ERR_NULL_POINTER, "NULL argument");
  if (num_steps < 0) return enf_set_error(ENF_ERR_BAD_DESC, "num_steps must be >= 0");
  if (method != ENF_ODE_EULER && method != ENF_ODE_RK4) return enf_set_error(ENF_ERR_BAD_DESC, "unknown method");   // solvers.py:151-152
  if ((rc = check_ptrs(d, w, workspace)) != ENF_OK) return rc;
  Ws Y = make_ws(d);
  if (workspace_bytes < (size_t)Y.total * sizeof(float)) return enf_set_error(ENF_ERR_WORKSPACE, "workspace too small");
  Run R; R.st = (cudaStream_t)stream; R.ws = (float*)workspace;
  cudaStream_t st = R.st;
  float* W = R.ws;
  const int T1 = num_steps + 1;
  const int64_t np = d.m * d.rec.P, na = d.m * d.L;
  auto store = [&](int step, const float* p, const float* a) {
    ode_store_traj_kernel<<<nblocks(np, 256), 256, 0, st>>>(d.Z, d.rec.P, T1, step, np, p, p_traj);
    ode_store_traj_kernel<<<nblocks(na, 256), 256, 0, st>>>(d.Z, d.L, T1, step, na, a, a_traj);
  };
  auto axpy = [&](int64_t n, const float* x, float c0, const float* k0, float c1, const float* k1, float c2, const float* k2, float c3,
                  const float* k3, float* y) { ode_axpy_kernel<<<nblocks(n, 256), 256, 0, st>>>(n, x, c0, k0, c1, k1, c2, k2, c3, k3, y); };
  float *cp = W + Y.tp, *ca = W + Y.ta;                    // stage inputs
  float *sp = W + Y.sp, *sa = W + Y.sa;                    // current state (the trajectory is [B, T+1, Z, .]: not contiguous per step)
  float* kp[4]; float* ka[4];
  for (int i = 0; i < 4; ++i) { kp[i] = W + Y.kp[i]; ka[i] = W + Y.ka[i]; }
  cudaMemcpyAsync(sp, p0, np * sizeof(float), cudaMemcpyDeviceToDevice, st);
  cudaMemcpyAsync(sa, a0, na * sizeof(float), cudaMemcpyDeviceToDevice, st);
  store(0, sp, sa);
  for (int i = 0; i < num_steps; ++i) {
    if (method == ENF_ODE_EULER) {                           // solvers.py:73-88
      if ((rc = forward(d, Y, *w, sp, sa, kp[0], ka[0], R)) != ENF_OK) return rc;
      axpy(np, sp, h, kp[0], 0, nullptr, 0, nullptr, 0, nullptr, sp);
      axpy(na, sa, h, ka[0], 0, nullptr, 0, nullptr, 0, nullptr, sa);
    } else {                                                 // solvers.py:91-108
      if ((rc = forward(d, Y, *w, sp, sa, kp[0], ka[0], R)) != ENF_OK) return rc;
      axpy(np, sp, 0.5f * h, kp[0], 0, nullptr, 0, nullptr, 0, nullptr, cp); axpy(na, sa, 0.5f * h, ka[0], 0, nullptr, 0, nullptr, 0, nullptr, ca);
      if ((rc = forward(d, Y, *w, cp, ca, kp[1], ka[1], R)) != ENF_OK) return rc;
      axpy(np, sp, 0.5f * h, kp[1], 0, nullptr, 0, nullptr, 0, nullptr, cp); axpy(na, sa, 0.5f * h, ka[1], 0, nullptr, 0, nullptr, 0, nullptr, ca);
      if ((rc = forward(d, Y, *w, cp, ca, kp[2], ka[2], R)) != ENF_OK) return rc;
      axpy(np, sp, h, kp[2], 0, nullptr, 0, nullptr, 0, nullptr, cp); axpy(na, sa, h, ka[2], 0, nullptr, 0, nullptr, 0, nullptr, ca);
      if ((rc = forward(d, Y, *w, cp, ca, kp[3], ka[3], R)) != ENF_OK) return rc;
      const float c = h / 6.f;
      axpy(np, sp, c, kp[0], 2.f * c, kp[1], 2.f * c, kp[2], c, kp[3], sp);
      axpy(na, sa, c, ka[0], 2.f * c, ka[1], 2.f * c, ka[2], c, ka[3], sa);
    }
    store(i + 1, sp, sa);
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return enf_set_error(ENF_ERR_CUDA, (std::string("CUDA error while enqueueing enf_ode_solve: ") + cudaGetErrorString(e)).c_str());
  return ENF_OK;
}

}  // extern "C"

// ---- MLPODE (mlp_ode.py:5-42) -----------------------------------------------------------------------------------------------
namespace {
struct MDims { int P, L, Hd, In; int64_t m; };
struct MWs {
  int64_t total = 0;
  int64_t take(int64_t n) { int64_t o = total; total += (n + 63) / 64 * 64; return o; }
  int64_t in, pre[2][3], act[2][3], g0, g1, g_in, g_in2;
};
int mlp_validate(const EnfMlpOdeDesc* D, MDims* o) {
  if (!D) return enf_set_error(ENF_ERR_NULL_POINTER, "desc is NULL");
  if (D->B <= 0 || D->Z <= 0 || D->L <= 0 || D->hidden <= 0) return enf_set_error(ENF_ERR_BAD_DESC, "B, Z, L, hidden must be positive");
  if (D->P != 2) return enf_set_error(ENF_ERR_UNSUPPORTED, "MLPODE emits a 2-component pose derivative (mlp_ode.py:27): P must be 2");
  if (D->reserved[0] || D->reserved[1] || D->reserved[2]) return enf_set_error(ENF_ERR_BAD_DESC, "reserved fields must be 0");
  o->P = D->P; o->L = D->L; o->Hd = D->hidden; o->In = D->P + D->L; o->m = (int64_t)D->B * D->Z;
  return ENF_OK;
}
MWs mlp_ws(const MDims& d) {
  MWs w;
  w.in = w.take(d.m * d.In);
  for (int k = 0; k < 2; ++k) for (int l = 0; l < 3; ++l) { w.pre[k][l] = w.take(d.m * d.Hd); w.act[k][l] = w.take(d.m * d.Hd); }
  w.g0 = w.take(d.m * d.Hd); w.g1 = w.take(d.m * d.Hd); w.g_in = w.take(d.m * d.In); w.g_in2 = w.take(d.m * d.In);
  return w;
}
// in = [p | a - 1]  (mlp_ode.py:35,38)
__global__ void mlpode_concat_kernel(int P, int L, int64_t m, const float* __restrict__ p, const float* __restrict__ a, float* __restrict__ in) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int In = P + L;
  if (t >= m * In) return;
  const int64_t r = t / In; const int c = (int)(t % In);
  in[t] = c < P ? p[r * P + c] : a[r * L + (c - P)] - 1.f;
}
__global__ void mlpode_split_kernel(int P, int L, int64_t m, const float* __restrict__ g_in, float* __restrict__ gp, float* __restrict__ ga) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int In = P + L;
  if (t >= m * In) return;
  const int64_t r = t / In; const int c = (int)(t % In);
  if (c < P) gp[r * P + c] = g_in[t]; else ga[r * L + (c - P)] = g_in[t];
}
int mlp_check(const EnfMlpOdeWeights* w, const void* workspace) {
  if (!w) return enf_set_error(ENF_ERR_NULL_POINTER, "weights are NULL");
  for (int l = 0; l < 4; ++l) if (!w->a_w[l] || !w->a_b[l] || !w->p_w[l] || !w->p_b[l]) return enf_set_error(ENF_ERR_NULL_POINTER, "a weight leaf is NULL");
  if (!workspace || ((uintptr_t)workspace & 255)) return enf_set_error(ENF_ERR_WORKSPACE, "workspace is NULL or not 256-byte aligned");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return enf_set_error(ENF_ERR_NO_DEVICE, "no CUDA device");
  return ENF_OK;
}
}  // namespace

extern "C" {

size_t enf_mlpode_workspace_bytes(const EnfMlpOdeDesc* desc) {
  MDims d;
  if (mlp_validate(desc, &d) != ENF_OK) return 0;
  return (size_t)mlp_ws(d).total * sizeof(float);
}

int enf_mlpode_fwd(const EnfMlpOdeDesc* desc, const EnfMlpOdeWeights* w, const float* p, const float* a, float* dp_dt, float* da_dt,
                   void* workspace, size_t workspace_bytes, enf_stream_t stream) {
  MDims d;
  int rc = mlp_validate(desc, &d);
  if (rc != ENF_OK) return rc;
  if (!p || !a || !dp_dt || !da_dt) return enf_set_error(ENF_ERR_NULL_POINTER, "NULL argument");
  if ((rc = mlp_check(w, workspace)) != ENF_OK) return rc;
  MWs Y = mlp_ws(d);
  if (workspace_bytes < (size_t)Y.total * sizeof(float)) return enf_set_error(ENF_ERR_WORKSPACE, "workspace too small: see enf_mlpode_workspace_bytes");
  Run R; R.st = (cudaStream_t)stream; R.ws = (float*)workspace;
  float* W = R.ws;
  mlpode_concat_kernel<<<nblocks(d.m * d.In, 256), 256, 0, R.st>>>(d.P, d.L, d.m, p, a, W + Y.in);
  for (int k = 0; k < 2; ++k) {                 // 0: mlp_a -> da/dt (L), 1: mlp_p -> dp/dt (2)
    const float* const* wk = k == 0 ? w->a_w : w->p_w;
    const float* const* bk = k == 0 ? w->a_b : w->p_b;
    const int nout = k == 0 ? d.L : 2;
    R.gemm(d.m, d.Hd, d.In, enf_mat(W + Y.in, d.In), enf_mat(wk[0], d.Hd), enf_mat(W + Y.pre[k][0], d.Hd), o_bias(bk[0], W + Y.act[k][0]));
    for (int l = 1; l < 3; ++l)
      R.gemm(d.m, d.Hd, d.Hd, enf_mat(W + Y.act[k][l - 1], d.Hd), enf_mat(wk[l], d.Hd), enf_mat(W + Y.pre[k][l], d.Hd), o_bias(bk[l], W + Y.act[k][l]));
    R.gemm(d.m, nout, d.Hd, enf_mat(W + Y.act[k][2], d.Hd), enf_mat(wk[3], nout), enf_mat(k == 0 ? da_dt : dp_dt, nout), o_bias(bk[3]));
  }
  if (R.failed) return enf_set_error(ENF_ERR_CUDA, "a GEMM of MLPODE could not be configured");
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return enf_set_error(ENF_ERR_CUDA, (std::string("CUDA error while enqueueing enf_mlpode_fwd: ") + cudaGetErrorString(e)).c_str());
  return ENF_OK;
}

int enf_mlpode_bwd(const EnfMlpOdeDesc* desc, const EnfMlpOdeWeights* w, const float* p, const float* a, const float* g_dp, const float* g_da,
                   const EnfMlpOdeWeightGrads* dW, float* gp, float* ga, void* workspace, size_t workspace_bytes, enf_stream_t stream) {
  MDims d;
  int rc = mlp_validate(desc, &d);
  if (rc != ENF_OK) return rc;
  if (!p || !a || !g_dp || !g_da || !gp || !ga) return enf_set_error(ENF_ERR_NULL_POINTER, "NULL argument");
  if ((rc = mlp_check(w, workspace)) != ENF_OK) return rc;
  MWs Y = mlp_ws(d);
  if (workspace_bytes < (size_t)Y.total * sizeof(float)) return enf_set_error(ENF_ERR_WORKSPACE, "workspace too small");
  Run R; R.st = (cudaStream_t)stream; R.ws = (float*)workspace;
  cudaStream_t st = R.st;
  float* W = R.ws;
  const bool wg = dW != nullptr;
  auto zero = [&](float* ptr, int64_t n) { cudaMemsetAsync(ptr, 0, n * sizeof(float), st); };
  for (int k = 0; k < 2; ++k) {
    const float* const* wk = k == 0 ? w->a_w : w->p_w;
    float* const* gwk = wg ? (k == 0 ? dW->a_w : dW->p_w) : nullptr;
    float* const* gbk = wg ? (k == 0 ? dW->a_b : dW->p_b) : nullptr;
    const int nout = k == 0 ? d.L : 2;
    const float* g_out = k == 0 ? g_da : g_dp;
    if (wg) {
      for (int l = 0; l < 4; ++l) if (!gwk[l] || !gbk[l]) return enf_set_error(ENF_ERR_NULL_POINTER, "a weight-gradient leaf is NULL");
      zero(gwk[0], (int64_t)d.In * d.Hd); zero(gwk[1], (int64_t)d.Hd * d.Hd); zero(gwk[2], (int64_t)d.Hd * d.Hd); zero(gwk[3], (int64_t)d.Hd * nout);
      zero(gbk[0], d.Hd); zero(gbk[1], d.Hd); zero(gbk[2], d.Hd); zero(gbk[3], nout);
      R.gemm(d.Hd, nout, (int)d.m, enf_mat(W + Y.act[k][2], 1, d.Hd), enf_mat(g_out, nout), enf_mat(gwk[3], nout), o_acc());
      R.launches += enf_launch_colsum(st, g_out, d.m, nout, nout, gbk[3], nullptr, 0);
    }
    float* g = W + Y.g0;
    float* g2 = W + Y.g1;
    R.gemm(d.m, d.Hd, nout, enf_mat(g_out, nout), enf_mat(wk[3], 1, nout), enf_mat(g, d.Hd), o_dgelu(W + Y.pre[k][2]));
    for (int l = 2; l >= 1; --l) {
      if (wg) {
        R.gemm(d.Hd, d.Hd, (int)d.m, enf_mat(W + Y.act[k][l - 1], 1, d.Hd), enf_mat(g, d.Hd), enf_mat(gwk[l], d.Hd), o_acc());
        R.launches += enf_launch_colsum(st, g, d.m, d.Hd, d.Hd, gbk[l], nullptr, 0);
      }
      R.gemm(d.m, d.Hd, d.Hd, enf_mat(g, d.Hd), enf_mat(wk[l], 1, d.Hd), enf_mat(g2, d.Hd), o_dgelu(W + Y.pre[k][l - 1]));
      float* t = g; g = g2; g2 = t;
    }
    if (wg) {
      R.gemm(d.In, d.Hd, (int)d.m, enf_mat(W + Y.in, 1, d.In), enf_mat(g, d.Hd), enf_mat(gwk[0], d.Hd), o_acc());
      R.launches += enf_launch_colsum(st, g, d.m, d.Hd, d.Hd, gbk[0], nullptr, 0);
    }
    if (k == 0) {
      R.gemm(d.m, d.In, d.Hd, enf_mat(g, d.Hd), enf_mat(wk[0], 1, d.Hd), enf_mat(W + Y.g_in, d.In));
    } else {                                    // second MLP: add to the first one's input cotangent
      R.gemm(d.m, d.In, d.Hd, enf_mat(g, d.Hd), enf_mat(wk[0], 1, d.Hd), enf_mat(W + Y.g_in2, d.In));
      R.launches += enf_launch_add(st, W + Y.g_in, W + Y.g_in, W + Y.g_in2, d.m * d.In);
    }
  }
  mlpode_split_kernel<<<nblocks(d.m * d.In, 256), 256, 0, st>>>(d.P, d.L, d.m, W + Y.g_in, gp, ga);
  if (R.failed) return enf_set_error(ENF_ERR_CUDA, "a GEMM of the MLPODE backward could not be configured");
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return enf_set_error(ENF_ERR_CUDA, (std::string("CUDA error while enqueueing enf_mlpode_bwd: ") + cudaGetErrorString(e)).c_str());
  return ENF_OK;
}

}  // extern "C"
