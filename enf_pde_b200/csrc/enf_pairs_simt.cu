// Fused (query, latent)-pair kernels, fp32 FMA path (EnfPrecision::ENF_PREC_FP32).
//
// One CTA owns a tile of TM = 32 coordinate queries of one field and loops over that field's Z
// latents.  For each latent the whole per-pair chain of equivariant_cross_attention.py:86-144 runs
// on [TM x d] activation tiles that never leave shared memory:
//     record -> invariants u, window w -> RFF_q -> W1_q,relu -> logits s (dot with folded U[z,h])
//                                       -> RFF_v -> W1_v,relu -> W' -> gelu,LN -> per head: W3[z,h] -> gelu,LN -> n
// forward : online softmax over latents, accumulating nbar = sum_z att * n      (never materialises
//           the queries x latents x embedding tensor)
// backward: recomputes the chain, then dgrad + wgrad per layer; per-latent gradient records
//           (dU, dkappa, dW3, db3, dLam, dsigma) and weight gradients are reduced with fp32 atomics.
// The folds (U, kappa, W', W3, b3) are DESIGN.md "Folds"; the math is tests/folded_model.py.
#include "enf_common.cuh"

namespace {

constexpr int TM = 32;        // query rows per CTA
constexpr int NT = 256;       // threads per CTA
constexpr int MAXH = 4;

template <int D> struct Cfg {
  static constexpr int LD = D + 4;                 // padded row stride (keeps 16B alignment)
  static constexpr int KC = D < 32 ? D : 32;       // weight rows staged per chunk
  static constexpr int CG = D / 4;                 // column groups (4 columns each)
  static constexpr int RG = NT / CG;               // row groups
  static constexpr int RM = (TM / RG) > 0 ? (TM / RG) : 1;   // rows per thread (GEMM)
  static constexpr int RK = (D / RG) > 0 ? (D / RG) : 1;     // k rows per thread (wgrad)
  static constexpr int BUF = TM * LD;
};

// Os[TM][D] (+)= act(As[TM][D] * Wg[D][D] + bias).   ACT: 0 none, 1 relu, 2 zero where mask<=0.
template <int D, int ACT, bool ACCUM>
__device__ __forceinline__ void tile_gemm(const float* __restrict__ As, const float* __restrict__ Wg, float* Os,
                                          const float* __restrict__ bias, const float* mask, float* Ws) {
  using C = Cfg<D>;
  const int tid = threadIdx.x;
  const int tx = tid % C::CG, rg = tid / C::CG;
  const int r0 = rg * C::RM;
  const bool active = r0 < TM;
  float acc[C::RM][4];
#pragma unroll
  for (int i = 0; i < C::RM; ++i) { acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f; }

  for (int kc = 0; kc < D; kc += C::KC) {
    // stage W[kc .. kc+KC) x D into shared memory (coalesced float4)
    const float4* src = reinterpret_cast<const float4*>(Wg + (size_t)kc * D);
    float4* dst = reinterpret_cast<float4*>(Ws);
    for (int e = tid; e < C::KC * D / 4; e += NT) dst[e] = __ldg(src + e);
    __syncthreads();
    if (active) {
#pragma unroll 2
      for (int k = 0; k < C::KC; k += 4) {
        float4 a[C::RM];
#pragma unroll
        for (int i = 0; i < C::RM; ++i) a[i] = *reinterpret_cast<const float4*>(As + (r0 + i) * C::LD + kc + k);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          float4 w = *reinterpret_cast<const float4*>(Ws + (k + kk) * D + tx * 4);
#pragma unroll
          for (int i = 0; i < C::RM; ++i) {
            float av = kk == 0 ? a[i].x : kk == 1 ? a[i].y : kk == 2 ? a[i].z : a[i].w;
            acc[i][0] = fmaf(av, w.x, acc[i][0]);
            acc[i][1] = fmaf(av, w.y, acc[i][1]);
            acc[i][2] = fmaf(av, w.z, acc[i][2]);
            acc[i][3] = fmaf(av, w.w, acc[i][3]);
          }
        }
      }
    }
    __syncthreads();
  }
  if (active) {
    float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (bias) b4 = __ldg(reinterpret_cast<const float4*>(bias + tx * 4));
#pragma unroll
    for (int i = 0; i < C::RM; ++i) {
      float* o = Os + (r0 + i) * C::LD + tx * 4;
      float4 v = make_float4(acc[i][0] + b4.x, acc[i][1] + b4.y, acc[i][2] + b4.z, acc[i][3] + b4.w);
      if (ACT == 1) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
      if (ACT == 2) {
        float4 m = *reinterpret_cast<const float4*>(mask + (r0 + i) * C::LD + tx * 4);
        v.x = m.x > 0.f ? v.x : 0.f; v.y = m.y > 0.f ? v.y : 0.f; v.z = m.z > 0.f ? v.z : 0.f; v.w = m.w > 0.f ? v.w : 0.f;
      }
      if (ACCUM) { float4 p = *reinterpret_cast<float4*>(o); v.x += p.x; v.y += p.y; v.z += p.z; v.w += p.w; }
      *reinterpret_cast<float4*>(o) = v;
    }
  }
  __syncthreads();
}

// dW[D][D] += As[TM][D]^T * Gs[TM][D]  (atomics);  db[D] += column sums of Gs (if db)
template <int D>
__device__ __forceinline__ void tile_wgrad(const float* __restrict__ As, const float* __restrict__ Gs, float* dW, float* db) {
  using C = Cfg<D>;
  const int tid = threadIdx.x;
  const int tx = tid % C::CG, kg = tid / C::CG;
  const int k0 = kg * C::RK;
  if (k0 < D) {
    float acc[C::RK][4];
#pragma unroll
    for (int i = 0; i < C::RK; ++i) { acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f; }
#pragma unroll 4
    for (int r = 0; r < TM; ++r) {
      float4 g = *reinterpret_cast<const float4*>(Gs + r * C::LD + tx * 4);
#pragma unroll
      for (int i = 0; i < C::RK; ++i) {
        float a = As[r * C::LD + k0 + i];
        acc[i][0] = fmaf(a, g.x, acc[i][0]);
        acc[i][1] = fmaf(a, g.y, acc[i][1]);
        acc[i][2] = fmaf(a, g.z, acc[i][2]);
        acc[i][3] = fmaf(a, g.w, acc[i][3]);
      }
    }
#pragma unroll
    for (int i = 0; i < C::RK; ++i) {
      float* o = dW + (size_t)(k0 + i) * D + tx * 4;
      atomicAdd(o + 0, acc[i][0]); atomicAdd(o + 1, acc[i][1]); atomicAdd(o + 2, acc[i][2]); atomicAdd(o + 3, acc[i][3]);
    }
  }
  if (db) {
    for (int j = tid; j < D; j += NT) {
      float s = 0.f;
#pragma unroll 8
      for (int r = 0; r < TM; ++r) s += Gs[r * C::LD + j];
      atomicAdd(db + j, s);
    }
  }
}

struct Smem {
  float* xi;      // [TM][8]
  float* u;       // [TM][8]
  float* w;       // [TM]
  float* s;       // [MAXH][TM]  logits / att
  float* m;       // [MAXH][TM]
  float* l;       // [MAXH][TM]
  float* aux;     // [MAXH][TM]  (bwd: ds)
  float* dd;      // [MAXH][TM]  (bwd: D = dnbar . nbar)
  float* du;      // [TM][8]
  float* dq;      // [TM][8]
  float* dsig;    // [TM]
  float* trstd;   // [TM]
  float* lam;     // [56]
  float* kap;     // [MAXH]
  float* Uz;      // [MAXH][D]
  float* omq;     // [6][D/2]
  float* omv;     // [6][D/2]
  float* lam2;    // [56]     frozen-relu mode: record of the mask poses
  float* u2;      // [TM][8]  frozen-relu mode: invariants against the mask poses
};

template <int D>
__device__ __forceinline__ float* carve_small(float* base, Smem& S) {
  float* p = base;
  S.xi = p; p += TM * 8;
  S.u = p; p += TM * 8;
  S.w = p; p += TM;
  S.s = p; p += MAXH * TM;
  S.m = p; p += MAXH * TM;
  S.l = p; p += MAXH * TM;
  S.aux = p; p += MAXH * TM;
  S.dd = p; p += MAXH * TM;
  S.du = p; p += TM * 8;
  S.dq = p; p += TM * 8;
  S.dsig = p; p += TM;
  S.trstd = p; p += TM;
  S.lam = p; p += 64;
  S.kap = p; p += 8;
  S.Uz = p; p += MAXH * D;
  S.omq = p; p += 6 * (D / 2);
  S.omv = p; p += 6 * (D / 2);
  S.lam2 = p; p += 64;
  S.u2 = p; p += TM * 8;
  return p;
}
template <int D> constexpr int small_floats() {
  return TM * 8 * 4 + TM * 3 + MAXH * TM * 5 + 64 + 8 + MAXH * D + 12 * (D / 2) + 64 + TM * 8;
}

// gamma(u) = [sin(2 pi u Omega) | cos(2 pi u Omega)]  (rff.py:84-93) into G[TM][D]
template <int D>
__device__ __forceinline__ void rff_features(const float* u, const float* om, int I, float* G) {
  constexpr int HD = D / 2;
  for (int e = threadIdx.x; e < TM * HD; e += NT) {
    int row = e / HD, j = e % HD;
    float proj = 0.f;
    for (int i = 0; i < I; ++i) proj = fmaf(u[row * 8 + i], om[i * HD + j], proj);
    float sn, cs;
    sincospif(2.f * proj, &sn, &cs);
    G[row * Cfg<D>::LD + j] = sn;
    G[row * Cfg<D>::LD + HD + j] = cs;
  }
}

// in-warp LayerNorm core of gelu(row): returns via out[], rstd
template <int D>
__device__ __forceinline__ float ln_gelu_row(const float* src, float* dst, int lane) {
  float s = 0.f, s2 = 0.f;
  for (int j = lane; j < D; j += 32) { float v = enf_gelu(src[j]); s += v; s2 += v * v; }
  s = warp_sum(s); s2 = warp_sum(s2);
  float mu = s * (1.f / D);
  float var = fmaxf(s2 * (1.f / D) - mu * mu, 0.f);
  float rstd = rsqrtf(var + 1e-6f);
  for (int j = lane; j < D; j += 32) { float v = enf_gelu(src[j]); dst[j] = (v - mu) * rstd; }
  return rstd;
}

// stage per-latent small vectors
template <int D>
__device__ __forceinline__ void stage_latent(const EnfPairParams& P, const Smem& S, int64_t bz) {
  const int tid = threadIdx.x;
  if (tid < ENF_LAM_SIZE) S.lam[tid] = P.lam[bz * ENF_LAM_SIZE + tid];
  if (tid < P.H) S.kap[tid] = P.kappa[bz * P.H + tid];
  for (int e = tid; e < P.H * D; e += NT) S.Uz[e] = P.U[bz * P.H * D + e];
}

// steps shared by forward and backward: invariants, q-path logits, v-path up to that = LN(gelu(tpre)).
// Buffers: Gq,H1q,Gv,H1v,Tpre,That (forward passes aliases: Gq=Gv=Tpre=That=bufA, H1q=H1v=bufB).
// Frozen-relu mode (P.lam_mask != null; the Hessian-vector products of the second-order outer gradient): the two relu layers
// use the activation PATTERN of the mask poses -- h = [pre(mask pose) > 0] * pre(evaluation pose) -- so that a finite difference
// of gradients along a latent direction differentiates the same piecewise-linear branch everywhere (what reverse-over-reverse
// autodiff does: relu'' = 0).  MQ / MV receive the mask poses' pre-activations ([TM][LD] each; tmpG is one more scratch tile);
// without the mode MQ = H1q and MV = H1v (callers test `> 0` on MQ / MV either way).
template <int D, bool KEEP>
__device__ __forceinline__ void pair_chain_common(const EnfPairParams& P, const Smem& S, int64_t bz,
                                                  float* Gq, float* H1q, float* Gv, float* H1v, float* Tpre,
                                                  float* That, float* Ws, float* MQ, float* MV, float* tmpG) {
  using C = Cfg<D>;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float scale = rsqrtf((float)D);
  const bool frozen = P.lam_mask != nullptr;
  stage_latent<D>(P, S, bz);
  if (frozen && tid < ENF_LAM_SIZE) S.lam2[tid] = P.lam_mask[bz * ENF_LAM_SIZE + tid];
  __syncthreads();
  if (tid < TM) {
    const float* xi = S.xi + tid * 8;
    const EnfPairRecord rec = pair_record<false>(P.rec, S.lam, xi, P.sigma ? P.sigma[bz] : 1.f);
#pragma unroll
    for (int r = 0; r < 6; ++r) {
      if (r < P.rec.I) {
        S.u[tid * 8 + r] = rec.u[r];
        if (frozen) S.u2[tid * 8 + r] = record_row(P.rec, S.lam2, xi, r);
      }
    }
    S.u[tid * 8 + 7] = rec.c;      // the raw cosine of a spherical window, for the backward (I <= 6 so slot 7 is free)
    S.w[tid] = rec.w;
  }
  __syncthreads();
  if (frozen) {
    rff_features<D>(S.u2, S.omq, P.rec.I, tmpG);
    __syncthreads();
    tile_gemm<D, 0, false>(tmpG, P.q_w1, MQ, P.q_b1, nullptr, Ws);            // pre-activations at the mask poses
  }
  rff_features<D>(S.u, S.omq, P.rec.I, Gq);
  __syncthreads();
  if (frozen) tile_gemm<D, 2, false>(Gq, P.q_w1, H1q, P.q_b1, MQ, Ws);
  else tile_gemm<D, 1, false>(Gq, P.q_w1, H1q, P.q_b1, nullptr, Ws);
  for (int r = warp; r < TM; r += NT / 32) {
    for (int h = 0; h < P.H; ++h) {
      float acc = 0.f;
      for (int j = lane; j < D; j += 32) acc = fmaf(H1q[r * C::LD + j], S.Uz[h * D + j], acc);
      acc = warp_sum(acc);
      if (lane == 0) S.s[h * TM + r] = scale * (acc + S.kap[h]) + S.w[r];
    }
  }
  if (!KEEP) __syncthreads();     // forward aliases Gq/Gv: everyone must be done reading H1q before it is reused
  if (frozen) {
    rff_features<D>(S.u2, S.omv, P.rec.I, tmpG);
    __syncthreads();
    tile_gemm<D, 0, false>(tmpG, P.v_w1, MV, P.v_b1, nullptr, Ws);
  }
  rff_features<D>(S.u, S.omv, P.rec.I, Gv);
  __syncthreads();
  if (frozen) tile_gemm<D, 2, false>(Gv, P.v_w1, H1v, P.v_b1, MV, Ws);
  else tile_gemm<D, 1, false>(Gv, P.v_w1, H1v, P.v_b1, nullptr, Ws);
  tile_gemm<D, 0, false>(H1v, P.Wp, Tpre, P.bp, nullptr, Ws);
  for (int r = warp; r < TM; r += NT / 32) {
    float rstd = ln_gelu_row<D>(Tpre + r * C::LD, That + r * C::LD, lane);
    if (lane == 0) S.trstd[r] = rstd;
  }
  __syncthreads();
}

// ------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------
template <int D>
__global__ void __launch_bounds__(NT, 1) pairs_fwd_kernel(EnfPairParams P) {
  using C = Cfg<D>;
  extern __shared__ __align__(16) float smem[];
  Smem S;
  float* p = carve_small<D>(smem, S);
  p = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(p) + 15) & ~uintptr_t(15));
  float* bufA = p; p += C::BUF;
  float* bufB = p; p += C::BUF;
  float* Ws = p; p += C::KC * D;
  float* acc = p; p += P.H * C::BUF;   // [H][TM][LD]
  float* bufMask = p;                  // frozen-relu mode only: [2][TM][LD] (mask pre-activations, scratch features)

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.y, c0 = blockIdx.x * TM;
  const int nv = min(TM, P.C - c0);
  const int H = P.H;

  for (int e = tid; e < TM * 8; e += NT) {
    int row = e >> 3;
    S.xi[e] = row < nv ? P.xi[(int64_t)b * P.xi_bs + (int64_t)(c0 + row) * 8 + (e & 7)] : 0.f;
  }
  for (int e = tid; e < P.rec.I * (D / 2); e += NT) { S.omq[e] = P.q_omega[e]; S.omv[e] = P.v_omega[e]; }
  for (int e = tid; e < MAXH * TM; e += NT) { S.m[e] = -INFINITY; S.l[e] = 0.f; }
  for (int e = tid; e < H * C::BUF; e += NT) acc[e] = 0.f;
  __syncthreads();

  for (int z = 0; z < P.Z; ++z) {
    const int64_t bz = (int64_t)b * P.Z + z;
    pair_chain_common<D, false>(P, S, bz, bufA, bufB, bufA, bufB, bufA, bufA, Ws, bufMask, bufMask, bufMask + C::BUF);
    // bufA now holds that = LN(gelu(tpre))
    for (int h = 0; h < H; ++h) {
      const int64_t bzh = bz * H + h;
      tile_gemm<D, 0, false>(bufA, P.W3 + bzh * D * D, bufB, P.b3 + bzh * D, nullptr, Ws);
      for (int r = warp; r < TM; r += NT / 32) {
        float* row = bufB + r * C::LD;
        ln_gelu_row<D>(row, row, lane);        // in place: n = LN(gelu(mpre))
        float m_old = S.m[h * TM + r], sv = S.s[h * TM + r];
        float m_new = fmaxf(m_old, sv);
        float corr = __expf(m_old - m_new);
        float pe = __expf(sv - m_new);
        float* a = acc + (h * TM + r) * C::LD;
        for (int j = lane; j < D; j += 32) a[j] = a[j] * corr + pe * row[j];
        __syncwarp();
        if (lane == 0) { S.m[h * TM + r] = m_new; S.l[h * TM + r] = S.l[h * TM + r] * corr + pe; }
      }
      __syncthreads();
    }
  }
  for (int r = warp; r < nv; r += NT / 32) {
    for (int h = 0; h < H; ++h) {
      float inv_l = 1.f / S.l[h * TM + r];
      const float* a = acc + (h * TM + r) * C::LD;
      float* o = P.nbar + (((int64_t)b * P.C + c0 + r) * H + h) * D;
      for (int j = lane; j < D; j += 32) o[j] = a[j] * inv_l;
      if (lane == 0) P.lse[((int64_t)b * P.C + c0 + r) * H + h] = S.m[h * TM + r] + logf(S.l[h * TM + r]);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------------------
template <int D>
__global__ void __launch_bounds__(NT, 1) pairs_bwd_kernel(EnfPairParams P) {
  using C = Cfg<D>;
  constexpr int HD = D / 2;
  extern __shared__ __align__(16) float smem[];
  Smem S;
  float* p = carve_small<D>(smem, S);
  p = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(p) + 15) & ~uintptr_t(15));
  float* Gq = p; p += C::BUF;
  float* H1q = p; p += C::BUF;
  float* Gv = p; p += C::BUF;
  float* H1v = p; p += C::BUF;
  float* Tpre = p; p += C::BUF;
  float* That = p; p += C::BUF;
  float* bufM = p; p += C::BUF;
  float* bufN = p; p += C::BUF;
  float* DT = p; p += C::BUF;
  float* Ws = p; p += C::KC * D;
  // frozen-relu mode: the mask poses' pre-activations of the two relu layers (otherwise the layers' own outputs serve as masks)
  float* MQ = P.lam_mask ? p : H1q;
  float* MV = P.lam_mask ? p + C::BUF : H1v;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.y, c0 = blockIdx.x * TM;
  const int nv = min(TM, P.C - c0);
  const int H = P.H;
  const float scale = rsqrtf((float)D);
  const float two_pi = 6.283185307179586f;

  for (int e = tid; e < TM * 8; e += NT) {
    int row = e >> 3;
    S.xi[e] = row < nv ? P.xi[(int64_t)b * P.xi_bs + (int64_t)(c0 + row) * 8 + (e & 7)] : 0.f;
  }
  for (int e = tid; e < P.rec.I * HD; e += NT) { S.omq[e] = P.q_omega[e]; S.omv[e] = P.v_omega[e]; }
  // lse (kept in S.m) and D = dnbar . nbar (S.dd) per (row, head)
  for (int r = warp; r < TM; r += NT / 32) {
    for (int h = 0; h < H; ++h) {
      float dsum = 0.f;
      if (r < nv) {
        const int64_t off = (((int64_t)b * P.C + c0 + r) * H + h) * D;
        for (int j = lane; j < D; j += 32) dsum = fmaf(P.dnbar[off + j], P.nbar[off + j], dsum);
      }
      dsum = warp_sum(dsum);
      if (lane == 0) {
        S.dd[h * TM + r] = dsum;
        S.m[h * TM + r] = r < nv ? P.lse[((int64_t)b * P.C + c0 + r) * H + h] : 0.f;
      }
    }
  }
  __syncthreads();

  float gxi[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};      // threads < TM: cotangent of the row's query record (P.g_xi only)
  for (int z = 0; z < P.Z; ++z) {
    const int64_t bz = (int64_t)b * P.Z + z;
    pair_chain_common<D, true>(P, S, bz, Gq, H1q, Gv, H1v, Tpre, That, Ws, MQ, MV, bufM);

    // ---- heads: recompute n, softmax weights, ds, dmpre; wgrad dW3/db3; dgrad into DT ------------
    for (int h = 0; h < H; ++h) {
      const int64_t bzh = bz * H + h;
      tile_gemm<D, 0, false>(That, P.W3 + bzh * D * D, bufM, P.b3 + bzh * D, nullptr, Ws);
      for (int r = warp; r < TM; r += NT / 32) {
        float* mrow = bufM + r * C::LD;
        float* nrow = bufN + r * C::LD;
        float rstd = ln_gelu_row<D>(mrow, nrow, lane);                 // n
        const bool valid = r < nv;
        float sv = S.s[h * TM + r];
        if (P.slog && valid) sv = P.slog[(((int64_t)b * P.Z + z) * P.C + c0 + r) * H + h];   // the forward's own logits
        float att = valid ? __expf(sv - S.m[h * TM + r]) : 0.f;
        const float* dnb = P.dnbar + (((int64_t)b * P.C + c0 + (valid ? r : 0)) * H + h) * D;
        float dotn = 0.f, m1 = 0.f;
        for (int j = lane; j < D; j += 32) {
          float dv = valid ? dnb[j] : 0.f;
          dotn = fmaf(dv, nrow[j], dotn);
          m1 += dv;
        }
        dotn = warp_sum(dotn); m1 = warp_sum(m1);
        // dn = att*dnbar ; LN-core backward needs mean(dn) and mean(dn*n)
        float mean1 = att * m1 * (1.f / D), mean2 = att * dotn * (1.f / D);
        for (int j = lane; j < D; j += 32) {
          float dv = valid ? dnb[j] : 0.f;
          float nj = nrow[j];
          float dg = rstd * (att * dv - mean1 - nj * mean2);
          nrow[j] = valid ? dg * enf_gelu_grad(mrow[j]) : 0.f;        // dmpre (in place over n)
        }
        if (lane == 0) S.aux[h * TM + r] = valid ? att * (dotn - S.dd[h * TM + r]) : 0.f;   // ds
      }
      __syncthreads();
      tile_wgrad<D>(That, bufN, P.g_W3 + bzh * D * D, P.g_b3 + bzh * D);
      if (h == 0) tile_gemm<D, 0, false>(bufN, P.W3T + bzh * D * D, DT, nullptr, nullptr, Ws);
      else        tile_gemm<D, 0, true>(bufN, P.W3T + bzh * D * D, DT, nullptr, nullptr, Ws);
    }
    // ---- dtpre = LNbwd(dthat) * gelu'(tpre)  (in place in DT) ------------------------------------
    for (int r = warp; r < TM; r += NT / 32) {
      float* drow = DT + r * C::LD;
      const float* th = That + r * C::LD;
      float m1 = 0.f, m2 = 0.f;
      for (int j = lane; j < D; j += 32) { m1 += drow[j]; m2 = fmaf(drow[j], th[j], m2); }
      m1 = warp_sum(m1) * (1.f / D); m2 = warp_sum(m2) * (1.f / D);
      float rstd = S.trstd[r];
      for (int j = lane; j < D; j += 32)
        drow[j] = rstd * (drow[j] - m1 - th[j] * m2) * enf_gelu_grad(Tpre[r * C::LD + j]);
    }
    __syncthreads();
    tile_wgrad<D>(H1v, DT, P.g_Wp, P.g_bp);
    tile_gemm<D, 2, false>(DT, P.WpT, bufM, nullptr, MV, Ws);                   // dzv = (dtpre Wp^T) * [h1v > 0]
    tile_wgrad<D>(Gv, bufM, P.g_v_w1, P.g_v_b1);
    tile_gemm<D, 0, false>(bufM, P.v_w1T, bufN, nullptr, nullptr, Ws);          // d gamma_v
    // du from the value embedding
    for (int r = warp; r < TM; r += NT / 32) {
      float part[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      for (int j = lane; j < HD; j += 32) {
        float dproj = Gv[r * C::LD + HD + j] * bufN[r * C::LD + j] - Gv[r * C::LD + j] * bufN[r * C::LD + HD + j];
        for (int i = 0; i < P.rec.I; ++i) part[i] = fmaf(dproj, S.omv[i * HD + j], part[i]);
      }
      for (int i = 0; i < P.rec.I; ++i) {
        float v = warp_sum(part[i]);
        if (lane == 0) S.du[r * 8 + i] = two_pi * v;
      }
    }
    // ---- query path: dzq = scale * sum_h ds_h U_h * [h1q > 0] ; dU, dkappa ------------------------
    for (int e = tid; e < TM * D; e += NT) {
      int r = e / D, i = e % D;
      float v = 0.f;
      for (int h = 0; h < H; ++h) v = fmaf(S.aux[h * TM + r], S.Uz[h * D + i], v);
      bufM[r * C::LD + i] = MQ[r * C::LD + i] > 0.f ? scale * v : 0.f;
    }
    for (int e = tid; e < H * D; e += NT) {
      int h = e / D, i = e % D;
      float v = 0.f;
#pragma unroll 8
      for (int r = 0; r < TM; ++r) v = fmaf(S.aux[h * TM + r], H1q[r * C::LD + i], v);
      atomicAdd(P.g_U + bz * H * D + e, scale * v);
    }
    if (tid < H) {
      float v = 0.f;
      for (int r = 0; r < TM; ++r) v += S.aux[tid * TM + r];
      atomicAdd(P.g_kappa + bz * H + tid, scale * v);
    }
    __syncthreads();
    tile_wgrad<D>(Gq, bufM, P.g_q_w1, P.g_q_b1);
    tile_gemm<D, 0, false>(bufM, P.q_w1T, bufN, nullptr, nullptr, Ws);          // d gamma_q
    for (int r = warp; r < TM; r += NT / 32) {
      float part[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      for (int j = lane; j < HD; j += 32) {
        float dproj = Gq[r * C::LD + HD + j] * bufN[r * C::LD + j] - Gq[r * C::LD + j] * bufN[r * C::LD + HD + j];
        for (int i = 0; i < P.rec.I; ++i) part[i] = fmaf(dproj, S.omq[i * HD + j], part[i]);
      }
      for (int i = 0; i < P.rec.I; ++i) {
        float v = warp_sum(part[i]);
        if (lane == 0) S.du[r * 8 + i] += two_pi * v;
      }
    }
    __syncthreads();
    // ---- invariants / window backward: cotangent of each record row, then reduce over the tile ----
    if (tid < TM) {
      const int t = tid;
      EnfPairRecord rec;
#pragma unroll
      for (int r = 0; r < 6; ++r) rec.u[r] = S.u[t * 8 + r];
      rec.w = S.w[t]; rec.c = S.u[t * 8 + 7];
      float du[6];
      for (int i = 0; i < 6; ++i) du[i] = i < P.rec.I ? S.du[t * 8 + i] : 0.f;
      float dw = 0.f;
      for (int h = 0; h < H; ++h) dw += S.aux[h * TM + t];
      float dq[ENF_R_LAM], dsg;
      record_adjoint(P.rec, rec, du, dw, P.sigma ? P.sigma[bz] : 1.f, dq, dsg);
#pragma unroll
      for (int r = 0; r < ENF_R_LAM; ++r) S.dq[t * 8 + r] = dq[r];
      S.dsig[t] = dsg;
      if (P.g_xi) {
        // cotangent of this row's QUERY record (self-attention: the queries are poses too, SURVEY 8f-4)
        record_xi_cotangent(P.rec, S.lam, S.xi + t * 8, dq, 0, gxi);
        record_xi_cotangent(P.rec, S.lam, S.xi + t * 8, dq, 1, gxi + 4);
      }
    }
    __syncthreads();
    if (tid < ENF_LAM_SIZE) {
      int r = tid / ENF_F_XI, f = tid % ENF_F_XI;
      float v = 0.f;
      for (int t = 0; t < TM; ++t) v = fmaf(S.dq[t * 8 + r], S.xi[t * 8 + f], v);
      atomicAdd(P.g_lam + bz * ENF_LAM_SIZE + tid, v);
    } else if (tid == 64 && P.rec.win_kind != ENF_WIN_NONE) {
      float v = 0.f;
      for (int t = 0; t < TM; ++t) v += S.dsig[t];
      atomicAdd(P.g_sigma + bz, v);
    }
    __syncthreads();
  }
  if (P.g_xi && tid < nv) {
    float* o = P.g_xi + ((int64_t)b * P.C + c0 + tid) * ENF_F_XI;
#pragma unroll
    for (int f = 0; f < 8; ++f) o[f] = gxi[f];
  }
}

template <int D> size_t fwd_smem(int H, bool frozen) {
  return (size_t)(small_floats<D>() + 4 + (2 + (frozen ? 2 : 0)) * Cfg<D>::BUF + Cfg<D>::KC * D + H * Cfg<D>::BUF) * sizeof(float);
}
template <int D> size_t bwd_smem(bool frozen) {
  return (size_t)(small_floats<D>() + 4 + (9 + (frozen ? 2 : 0)) * Cfg<D>::BUF + Cfg<D>::KC * D) * sizeof(float);
}

template <int D>
int launch_fwd(cudaStream_t st, const EnfPairParams& p) {
  size_t smem = fwd_smem<D>(p.H, p.lam_mask != nullptr);
  if (cudaFuncSetAttribute(pairs_fwd_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return -1;
  dim3 grid((p.C + TM - 1) / TM, p.B);
  pairs_fwd_kernel<D><<<grid, NT, smem, st>>>(p);
  return 1;
}
template <int D>
int launch_bwd(cudaStream_t st, const EnfPairParams& p) {
  size_t smem = bwd_smem<D>(p.lam_mask != nullptr);
  if (cudaFuncSetAttribute(pairs_bwd_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return -1;
  dim3 grid((p.C + TM - 1) / TM, p.B);
  pairs_bwd_kernel<D><<<grid, NT, smem, st>>>(p);
  return 1;
}

}  // namespace

int enf_launch_pairs_fwd_simt(cudaStream_t st, int d, const EnfPairParams& p) {
  switch (d) {
    case 16: return launch_fwd<16>(st, p);
    case 32: return launch_fwd<32>(st, p);
    case 64: return launch_fwd<64>(st, p);
    case 128: return launch_fwd<128>(st, p);
  }
  return -1;
}
int enf_launch_pairs_bwd_simt(cudaStream_t st, int d, const EnfPairParams& p) {
  switch (d) {
    case 16: return launch_bwd<16>(st, p);
    case 32: return launch_bwd<32>(st, p);
    case 64: return launch_bwd<64>(st, p);
    case 128: return launch_bwd<128>(st, p);
  }
  return -1;
}
