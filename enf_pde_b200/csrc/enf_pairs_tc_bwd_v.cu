// Fused (query, latent)-pair BACKWARD, kernel B: the bottom of the VALUE path (EnfPrecision::ENF_PREC_BF16, d = 128).
// Runs after kernel A (enf_pairs_tc_bwd.cu), before kernel C (enf_pairs_tc_bwd_q.cu).
//
// Persistent CTAs walk (field, latent) items; per item they walk the field's query tiles (128 rows each):
//     S1  gamma_v (hi | lo fp16 split) from the RFF phases the tensor core left in TMEM
//     M1  T    = gamma_v W1_v                 (3-term split product: the relu mask decides whole gradient entries)
//     E3  (in M1's shadow) dtpre = (dthat - mean(dthat) - that mean(dthat that)) * (rstd gelu'(tpre))   -> operand tile
//         = LayerNorm / gelu backward from three fp16 streams: dthat (kernel A) and the forward's stashes `that`, `dgr` (+ rstd per row);
//         nothing of the layer above h1v is recomputed here (no h1v W' product, no tanh)
//     E2  h1v  = relu(T + b1v)  -> operand tile ; mask bits stay in a register
//     M3  T    = dtpre W'^T     dW' += h1v^T dtpre     db' += dtpre^T 1
//     E4  dzv  = T [h1v > 0]                                                                    -> operand tile
//     M4  T    = dzv W1_v^T (d gamma_v)     dW1_v += gamma_v^T dzv     db1v += dzv^T 1
//     S3  dproj_j = cos_j dsin_j - sin_j dcos_j   (thread-local: a thread owns sin AND cos of its 16 frequencies) -> tile
//     M5  du = dproj Omega^T                  (N = 16: [Omega_hi | Omega_lo])
//     S4  (one thread per row, overlapped with the next tile's M1)  du -> duv[b,z,c,:] for kernel C
// Column sums over query rows (bias gradients) are `tile^T x 1` MMAs against a constant side operand.  The three
// shared-weight accumulators (dW', dW1_v, their biases) live in TMEM for the CTA's whole life and are flushed once,
// so the kernel issues 148 x 2 x d^2 global atomics in total.
#include <cuda_fp16.h>

#include "enf_pairs_tc_common.cuh"

namespace {

using namespace tcp;

template <int D> struct VCfg {
  static constexpr int NQ = D / 32;
  static constexpr int NT = ROWS * NQ;
  static constexpr int HD = D / 2;
  static constexpr uint32_t WIMG = wimg_bytes<D>();
  static constexpr uint32_t WBLK = D * 128;
  static constexpr uint32_t ABLK = ROWS * 128;
  static constexpr uint32_t ATILE = atile_bytes<D>();
  static constexpr int TMEM_NEED = 3 * D + 64 + 48;           // T | dW' | dW1_v | phases (64) | db' | db1v | du (16 each)
  static constexpr int TMEM_COLS = TMEM_NEED <= 256 ? 256 : 512;
  static constexpr int kDuCq = NQ > 1 ? 1 : 0;                // the row's thread that hands du to kernel C
  static constexpr uint32_t OFF_W = 0;                         // W1_v image, W1_v low image, W' image
  static constexpr uint32_t OFF_GHI = 3 * WIMG;                // gamma_v hi
  static constexpr uint32_t OFF_X = OFF_GHI + ATILE;           // gamma_v lo -> h1v -> dproj
  static constexpr uint32_t OFF_DT = OFF_X + ATILE;            // dtpre -> dzv
  static constexpr uint32_t OFF_ONE = OFF_DT + ATILE;          // side operand: K-major [16][128 rows], row 0 = ones
  static constexpr uint32_t OFF_U = OFF_ONE + 2 * 2048;        // projection operand (invariants), 2 atoms
  static constexpr uint32_t OFF_OM = OFF_U + 2 * kProjAtom;    // Omega_v projection image, 1 atom
  static constexpr uint32_t OFF_OMT = OFF_OM + kProjAtom;      // Omega_v^T image for du, [16][64]
  static constexpr uint32_t OFF_F = OFF_OMT + 2048;
  static constexpr int F_TOTAL = 64 /*lam*/ + 2 * D /*b1v | bp*/ + NQ * ROWS * 4 /*row exchange*/;
  static constexpr uint32_t SMEM_BYTES = OFF_F + F_TOTAL * 4 + 128 + 1024;
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
};

__device__ __forceinline__ void load_scale_v(const float* gmax, float& gs, float& inv_gs) {
  float m = *gmax;
  int e = 0;
  const bool ok = m > 0.f && isfinite(m);
  if (ok) frexpf(m, &e);
  gs = ok ? ldexpf(1.f, 4 - e) : 1.f;
  inv_gs = 1.f / gs;
}

// D[D x 16] (+)= Act^T S : Act = [128 rows][D] activation tile read MN-major (M = feature), S = K-major [16][128 rows]
template <int D>
__device__ __forceinline__ void issue_colsum(uint32_t d_tmem, uint32_t act_addr, uint32_t one_addr, uint32_t ablk, uint32_t accumulate) {
  constexpr uint32_t idesc = tc::make_idesc(wgrad_m<D>(), 16, tc::kOperandFmt, 1, 0);
#pragma unroll
  for (int kk = 0; kk < ROWS / 16; ++kk)
    tc::mma_f16(d_tmem, tc::desc_mnmajor(act_addr + kk * 2048, ablk), tc::desc_kmajor(one_addr + (kk >> 2) * 2048 + (kk & 3) * 32), idesc,
                (kk > 0) | accumulate);
}
// D[128 x 16] = Dp[128 rows][HD <= 64] (K-major, first feature block) * OmT[16][HD] (K-major)
template <int HD>
__device__ __forceinline__ void issue_du_v(uint32_t d_tmem, uint32_t a_addr, uint32_t b_addr) {
  constexpr uint32_t idesc = tc::make_idesc(ROWS, 16, tc::kOperandFmt, 0, 0);
#pragma unroll
  for (int kk = 0; kk < HD / 16; ++kk) tc::mma_f16(d_tmem, tc::desc_kmajor(a_addr + kk * 32), tc::desc_kmajor(b_addr + kk * 32), idesc, kk > 0);
}

template <int D>
__global__ void __launch_bounds__(VCfg<D>::NT, D == 32 ? 2 : 1) pairs_bwd_tc_v_kernel(EnfPairTcBwdParams P) {
  using C = VCfg<D>;
  constexpr int HD = C::HD;
  constexpr int MMA_TID = C::NT - 128;                // lane 0 of the first warp of the last column quarter
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sW = base + C::OFF_W;
  uint8_t* sGhi = base + C::OFF_GHI;
  uint8_t* sX = base + C::OFF_X;
  uint8_t* sDt = base + C::OFF_DT;
  uint8_t* sOne = base + C::OFF_ONE;
  uint8_t* sU = base + C::OFF_U;
  uint8_t* sOm = base + C::OFF_OM;
  uint8_t* sOmT = base + C::OFF_OMT;
  float* f = reinterpret_cast<float*>(base + C::OFF_F);
  float* s_lam = f; f += 64;
  float* s_bias = f; f += 2 * D;                      // b1v | bp
  float* s_exch = f; f += C::NQ * ROWS * 4;          // one buffer: a single exchange per tile, block barriers in between
  uint64_t* bars = reinterpret_cast<uint64_t*>(f);
  uint64_t *bar_w = bars, *bar_p = bars + 1, *bar_g1 = bars + 2, *bar_t = bars + 3, *bar_g3 = bars + 4, *bar_g3b = bars + 5,
           *bar_g4 = bars + 6, *bar_u = bars + 7;
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bars + 8);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int lq = warp & 3, cq = warp >> 2;
  const int row = lq * 32 + lane, col0 = cq * 32;

  if (tid == 0) {
    for (int i = 0; i < 8; ++i) tc::mbar_init(bars + i, 1);
    tc::mbar_fence_init();
  }
  if (warp == 0) tc::tmem_alloc<C::TMEM_COLS>(s_tmem);
  for (int e = tid; e < D; e += C::NT) { s_bias[e] = P.v_b1[e]; s_bias[D + e] = P.bp[e]; }
  {
    uint4* z4 = reinterpret_cast<uint4*>(sOne);       // One, U, Om, OmT are contiguous
    for (int e = tid; e < (int)(C::OFF_F - C::OFF_ONE) / 16; e += C::NT) z4[e] = make_uint4(0u, 0u, 0u, 0u);
  }
  float gs, inv_gs;
  load_scale_v(P.gmax, gs, inv_gs);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tm = *s_tmem;
  const uint32_t tT = tm, tWp = tm + D, tW1 = tm + 2 * D, tP = tm + 3 * D, tS1 = tP + 64, tS2 = tS1 + 16, tDu = tS2 + 16;
  const uint32_t lane_off = (uint32_t)(lq * 32) << 16;
  const uint32_t my_t = lane_off + col0;
  if (tid == MMA_TID) {
    tc::mbar_expect_tx(bar_w, 3 * C::WIMG);
    tc::bulk_g2s(sW, P.img_v_w1, C::WIMG, bar_w);
    tc::bulk_g2s(sW + C::WIMG, P.img_v_w1_lo, C::WIMG, bar_w);
    tc::bulk_g2s(sW + 2 * C::WIMG, P.img_Wp, C::WIMG, bar_w);
  }
  const uint32_t aW = tc::smem_u32(sW), aWlo = aW + C::WIMG, aWp = aW + 2 * C::WIMG, aGhi = tc::smem_u32(sGhi), aX = tc::smem_u32(sX),
                 aDt = tc::smem_u32(sDt), aOne = tc::smem_u32(sOne), aU = tc::smem_u32(sU), aOm = tc::smem_u32(sOm),
                 aOmT = tc::smem_u32(sOmT);
  // constant side operand: K-major [16][128 rows]; row 0 (the only non-zero output column) = ones
  if (tid < ROWS) {
    const int k = tid;                                 // query row = K index
    *reinterpret_cast<__half*>(sOne + (k >> 6) * 2048 + ((((k & 63) >> 3) ^ 0) << 4) + (k & 7) * 2) = __float2half_rn(1.f);
  }
  // Omega images: projection operand (phases) and its transpose for du, both as a two-term fp16 split of 2 pi Omega
  proj_build_omega(sOm, 0, P.v_omega, P.rec.I, HD, tid, C::NT);
  for (int e = tid; e < P.rec.I * HD; e += C::NT) {
    const int i = e / HD, j = e % HD;
    const float val = 6.283185307179586f * P.v_omega[e];
    const __half hi = __float2half_rn(val);
    const __half lo = __float2half_rn(val - __half2float(hi));
    auto off = [&](int n) { return (uint32_t)((n >> 3) * 1024 + (n & 7) * 128 + ((((j >> 3) ^ (n & 7))) << 4) + (j & 7) * 2); };
    *reinterpret_cast<__half*>(sOmT + off(i)) = hi;
    *reinterpret_cast<__half*>(sOmT + off(6 + i)) = lo;
  }

  const int ntiles = (P.C + ROWS - 1) / ROWS;
  const int nitems = P.B * P.Z;
  uint32_t it = 0;                                     // tiles processed by this CTA (barrier parities)
  int xw = 0;

  for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
    const int64_t bz = item;
    const int b = item / P.Z;
    __syncthreads();                                   // the previous item's last side work is done with s_lam
    if (tid < ENF_LAM_SIZE) s_lam[tid] = P.lam[bz * ENF_LAM_SIZE + tid];
    const float sigma = P.sigma ? P.sigma[bz] : 1.f;
    __syncthreads();

    auto load_xi = [&](int ct, float* xi_r) {
#pragma unroll
      for (int k = 0; k < 8; ++k) xi_r[k] = 0.f;
      if (ct * ROWS + row < P.C) {
        const float4* src = reinterpret_cast<const float4*>(P.xi + (int64_t)b * P.xi_bs + (int64_t)(ct * ROWS + row) * 8);
        float4 a = __ldg(src), c = __ldg(src + 1);
        xi_r[0] = a.x; xi_r[1] = a.y; xi_r[2] = a.z; xi_r[3] = a.w; xi_r[4] = c.x; xi_r[5] = c.y; xi_r[6] = c.z; xi_r[7] = c.w;
      }
    };
    auto write_invariants = [&](const float* xi_r) {
      const EnfPairRecord rec = pair_record<true>(P.rec, s_lam, xi_r, sigma);
      proj_write_u(sU, row, rec.u, P.rec.I);
    };
    // one thread per row: du of tile ct (value path) -> duv for kernel C
    auto store_du = [&](int ct, uint32_t par_u) {
      tc::mbar_wait(bar_u, par_u);
      tc::tc_fence_after();
      float d16[16];
      tc::tmem_ld16(tDu + lane_off, d16);
      tc::tmem_ld_wait();
      if (ct * ROWS + row < P.C) {
        float du[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) du[i] = (i < 6 && i < P.rec.I) ? d16[i] + d16[6 + i] : 0.f;
        float4* dst = reinterpret_cast<float4*>(P.duv + (bz * P.C + ct * ROWS + row) * 8);
        dst[0] = make_float4(du[0], du[1], du[2], du[3]);
        dst[1] = make_float4(du[4], du[5], du[6], du[7]);
      }
    };

    if (cq == 0) {
      float xi0[8];
      load_xi(0, xi0);
      write_invariants(xi0);
    }
    tc::fence_proxy_async();
    __syncthreads();
    if (tid == MMA_TID) {
      tc::tc_fence_after();
      issue_proj(tP, aU, aOm, HD);
      tc::mma_commit(bar_p);
    }

    for (int ct = 0; ct < ntiles; ++ct, ++it) {
      const uint32_t par = it & 1;
      const int c0 = ct * ROWS;
      const bool valid = c0 + row < P.C;
      const int64_t pr = bz * P.C + c0 + row;
      // my 32 columns of the three fp16 streams of E3: cotangent of that (kernel A), that and rstd * gelu' (stashed by the
      // forward); requested here, first touched after S1
      uint4 dthq[4], dgq[4];
      const int64_t chunked = ((bz * ntiles + ct) * C::NQ + cq) * 4 * ROWS + row;
      {
        const uint4* src = reinterpret_cast<const uint4*>(P.dthat) + chunked;
#pragma unroll
        for (int q = 0; q < 4; ++q) dthq[q] = valid ? __ldg(src + q * ROWS) : make_uint4(0u, 0u, 0u, 0u);
      }
      if (it > 0) {                                        // every MMA of the previous tile is done with the operand tiles
        tc::mbar_wait(bar_u, (it - 1) & 1);
        tc::tc_fence_after();
      }
      if (tid == MMA_TID) {                                // the `that` operand image of this tile -> the (free) dtpre tile: E3 reads
        tc::mbar_expect_tx(bar_t, C::ATILE);               // its own chunks from there and overwrites them in place
        tc::bulk_g2s(sDt, P.that_img + (size_t)(bz * ntiles + ct) * C::ATILE, C::ATILE, bar_t);
      }
      if (cq == C::kDuCq && ct > 0) store_du(ct - 1, (it - 1) & 1);      // previous tile's du -> duv (the item's last tile: at its flush)
      // ---- S1: gamma_v hi / lo ---------------------------------------------------------------------------------
      tc::mbar_wait(bar_p, par);
      tc::tc_fence_after();
      // sin half first: the K-steps over the sin features (3 split terms) are issued as soon as that half is written
      // (named barrier 5: the issuing warp syncs, the others arrive) and run in the shadow of the cos half
      constexpr int KH = D / 32;                           // K-steps (16 features) per half of gamma
      rff_half_from_proj<D, true, true>(tP + lane_off + 16 * cq, sGhi, sX, C::ABLK, row, 16 * cq);
      tc::fence_proxy_async();
      if (warp == (MMA_TID >> 5)) {
        tc::named_sync(5, C::NT);
        if (tid == MMA_TID) {
          if (it == 0) tc::mbar_wait(bar_w, 0);
          tc::tc_fence_after();
          issue_gemm_ksteps<D>(tT, aGhi, aW, C::ABLK, C::WBLK, 0, KH, 0);
          issue_gemm_ksteps<D>(tT, aX, aW, C::ABLK, C::WBLK, 0, KH, 1);
          issue_gemm_ksteps<D>(tT, aGhi, aWlo, C::ABLK, C::WBLK, 0, KH, 1);
        }
        __syncwarp();
      } else {
        tc::named_arrive(5, C::NT);
      }
      {                                                    // second stream of E3 (all CTAs reach their tile tops together: the
        const uint4* srg = P.dgr + chunked;                // requests are staggered so that they do not queue behind each other)
#pragma unroll
        for (int q = 0; q < 4; ++q) dgq[q] = valid ? __ldg(srg + q * ROWS) : make_uint4(0u, 0u, 0u, 0u);
      }
      const float trs = valid ? __ldg(P.trstd + (size_t)bz * ntiles * ROWS + c0 + row) : 0.f;
      rff_half_from_proj<D, true, false>(tP + lane_off + 16 * cq, sGhi, sX, C::ABLK, row, 16 * cq);
      tc::tc_fence_before();
      tc::fence_proxy_async();
      __syncthreads();
      if (tid == MMA_TID) {
        tc::tc_fence_after();
        issue_gemm_ksteps<D>(tT, aGhi, aW, C::ABLK, C::WBLK, KH, 2 * KH, 1);
        issue_gemm_ksteps<D>(tT, aX, aW, C::ABLK, C::WBLK, KH, 2 * KH, 1);
        issue_gemm_ksteps<D>(tT, aGhi, aWlo, C::ABLK, C::WBLK, KH, 2 * KH, 1);
        tc::mma_commit(bar_g1);
      }
      // ---- in the shadow of the 3-term GEMM: E3 and the next tile's invariants -----------------------------------------
      float xi_next[8];
      if (cq == 0 && ct + 1 < ntiles) load_xi(ct + 1, xi_next);      // requested now, used after E3
      {
        // LayerNorm backward needs the row sums  sum_j dth_j  and  sum_j dth_j that_j
        uint4 thq[4];
        tc::mbar_wait(bar_t, par);
        {
          const uint8_t* trow = sDt + (col0 >> 6) * C::ABLK;
#pragma unroll
          for (int q = 0; q < 4; ++q)
            thq[q] = valid ? *reinterpret_cast<const uint4*>(trow + tc::swz_chunk_off(row, ((col0 & 63) >> 3) + q)) : make_uint4(0u, 0u, 0u, 0u);
        }
        float st[2];
        {
          float2 s2 = tc::splat2(0.f), s3 = tc::splat2(0.f);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const __half2* hd = reinterpret_cast<const __half2*>(&dthq[q]);
            const __half2* ht = reinterpret_cast<const __half2*>(&thq[q]);
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              const float2 d = __half22float2(hd[t]);
              s2 = tc::fma2(d, __half22float2(ht[t]), s2); s3 = tc::add2(s3, d);
            }
          }
          st[0] = s2.x + s2.y; st[1] = s3.x + s3.y;
        }
        xw = 0;
        row_exchange<C::NQ, 2>(s_exch, xw, cq, row, lq, st);
        const float2 nm2 = tc::splat2(-st[0] * (1.f / D) * trs), nm1 = tc::splat2(-st[1] * (1.f / D) * trs), rs2 = tc::splat2(trs);
        // dtpre = rstd (dth - m1 - that m2) g'
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const __half2* hd = reinterpret_cast<const __half2*>(&dthq[q]);
          const __half2* ht = reinterpret_cast<const __half2*>(&thq[q]);
          const __half2* hg = reinterpret_cast<const __half2*>(&dgq[q]);
          float o[8];
#pragma unroll
          for (int t = 0; t < 4; ++t)
            tc::st2(o + 2 * t, tc::mul2(tc::fma2(__half22float2(ht[t]), nm2, tc::fma2(__half22float2(hd[t]), rs2, nm1)), __half22float2(hg[t])));
          tc::st_row8_bf16(sDt, C::ABLK, row, col0 + 8 * q, o);
        }
      }
      // next tile's invariants -> projection operand (tP was read by everyone before the barrier)
      if (cq == 0 && ct + 1 < ntiles) write_invariants(xi_next);
      // ---- E2: h1v, mask ---------------------------------------------------------------------------------------------
      float v[32];
      tc::mbar_wait(bar_g1, par);
      tc::tc_fence_after();
      tc::tmem_ld32(tT + my_t, v);
      tc::tmem_ld_wait();
      uint32_t neg = 0;                                    // bit j: pre-activation j is negative (sign bits, two integer ops per element)
#pragma unroll
      for (int c8 = 0; c8 < 32; c8 += 8) {
        float o[8];
        const float4 b0 = *reinterpret_cast<const float4*>(s_bias + col0 + c8);
        const float4 b1 = *reinterpret_cast<const float4*>(s_bias + col0 + c8 + 4);
        const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
        for (int t = 0; t < 8; ++t) {
          const float pre = v[c8 + t] + bv[t];
          o[t] = fmaxf(pre, 0.f);
          neg |= (__float_as_uint(pre) & 0x80000000u) >> (31 - (c8 + t));
        }
        tc::st_row8_bf16(sX, C::ABLK, row, col0 + c8, o);
      }
      tc::tc_fence_before();
      tc::fence_proxy_async();
      __syncthreads();
      if (tid == MMA_TID) {
        tc::tc_fence_after();
        issue_dgrad<D>(tT, aDt, aWp, C::ABLK, C::WBLK, 0);          // d h1v
        tc::mma_commit(bar_g3);
        if (P.g_Wp) {                                       // latents-only backward (dW = NULL): no shared-weight gradients
          issue_wgrad<D>(tWp, aX, aDt, C::ABLK, it > 0);            // dW' (per CTA)
          issue_colsum<D>(tS1, aDt, aOne, C::ABLK, it > 0);         // db' (per CTA)
        }
        tc::mma_commit(bar_g3b);                                    // (without them: fires with the dgrad, which reads dtpre too)
        if (ct + 1 < ntiles) {                             // phases of the next tile (sU was written before the barrier)
          issue_proj(tP, aU, aOm, HD);
          tc::mma_commit(bar_p);
        }
      }
      // ---- E4: dzv = d h1v [h1v > 0] ----------------------------------------------------------------------------------
      tc::mbar_wait(bar_g3, par);
      tc::tc_fence_after();
      tc::tmem_ld32(tT + my_t, v);
      tc::tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = ((neg >> j) & 1u) ? 0.f : v[j];
      tc::mbar_wait(bar_g3b, par);                         // the wgrad has finished reading dtpre: its tile takes dzv
#pragma unroll
      for (int c8 = 0; c8 < 32; c8 += 8) tc::st_row8_bf16(sDt, C::ABLK, row, col0 + c8, v + c8);
      tc::tc_fence_before();
      tc::fence_proxy_async();
      __syncthreads();
      if (tid == MMA_TID) {
        tc::tc_fence_after();
        issue_dgrad<D>(tT, aDt, aW, C::ABLK, C::WBLK, 0);           // d gamma_v
        tc::mma_commit(bar_g4);
        if (P.g_Wp) {
          issue_wgrad<D>(tW1, aGhi, aDt, C::ABLK, it > 0);          // dW1_v (per CTA)
          issue_colsum<D>(tS2, aDt, aOne, C::ABLK, it > 0);         // db1v (per CTA)
        }
      }
      // ---- S3: d gamma_v -> dproj (my 16 frequencies: sin columns j, cos columns HD + j) ---------------------------
      tc::mbar_wait(bar_g4, par);
      tc::tc_fence_after();
      {
        float dsn[16], dcs[16];
        tc::tmem_ld16(tT + lane_off + 16 * cq, dsn);
        tc::tmem_ld16(tT + lane_off + HD + 16 * cq, dcs);
        tc::tmem_ld_wait();
#pragma unroll
        for (int c8 = 0; c8 < 16; c8 += 8) {
          const int col = 16 * cq + c8;                              // sin feature `col`, cos feature HD + col
          const uint4 qs = *reinterpret_cast<const uint4*>(sGhi + tc::swz_chunk_off(row, col >> 3));
          const uint4 qc = *reinterpret_cast<const uint4*>(sGhi + ((HD + col) >> 6) * C::ABLK + tc::swz_chunk_off(row, ((HD + col) & 63) >> 3));
          const __half2* hs = reinterpret_cast<const __half2*>(&qs);
          const __half2* hc = reinterpret_cast<const __half2*>(&qc);
          float o[8];
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const float2 sn = __half22float2(hs[t]), cs = __half22float2(hc[t]);
            o[2 * t] = cs.x * dsn[c8 + 2 * t] - sn.x * dcs[c8 + 2 * t];
            o[2 * t + 1] = cs.y * dsn[c8 + 2 * t + 1] - sn.y * dcs[c8 + 2 * t + 1];
          }
          tc::st_row8_bf16(sX, C::ABLK, row, col, o);               // h1v's wgrad completed before E4 stored (bar_g3b)
        }
      }
      tc::tc_fence_before();
      tc::fence_proxy_async();
      __syncthreads();
      if (tid == MMA_TID) {
        tc::tc_fence_after();
        issue_du_v<HD>(tDu, aX, aOmT);
        tc::mma_commit(bar_u);
      }
    }
    // ---- item flush: the last tile's du ----------------------------------------------------------------------------
    if (cq == C::kDuCq) store_du(ntiles - 1, (it - 1) & 1);
  }
  // ---- CTA flush: shared-weight gradients ------------------------------------------------------------------------------
  if (it > 0) {
    tc::mbar_wait(bar_u, (it - 1) & 1);
    tc::tc_fence_after();
  }
  __syncthreads();
  tc::tc_fence_after();
  if (it > 0 && P.g_Wp) {
    const int wrow = wgrad_row<D>(row, lq, lane);      // accumulator row (input feature) of this thread
    float* dst[2] = {P.g_Wp, P.g_v_w1};
    const uint32_t src[2] = {tWp, tW1};
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      float v[32];
      tc::tmem_ld32(src[k] + my_t, v);
      tc::tmem_ld_wait();
      if (wrow >= 0) {
        float* o = dst[k] + (size_t)wrow * D + col0;
#pragma unroll
        for (int j = 0; j < 32; ++j) atomicAdd(o + j, v[j] * inv_gs);
      }
    }
    if (cq == 0) {
      float d16[16];
      tc::tmem_ld16(tS1 + lane_off, d16);
      tc::tmem_ld_wait();
      if (wrow >= 0) atomicAdd(P.g_bp + wrow, d16[0] * inv_gs);
      tc::tmem_ld16(tS2 + lane_off, d16);
      tc::tmem_ld_wait();
      if (wrow >= 0) atomicAdd(P.g_v_b1 + wrow, d16[0] * inv_gs);
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc<C::TMEM_COLS>(tm);
}

template <int D>
int launch_v(cudaStream_t st, const EnfPairTcBwdParams& p) {
  using C = VCfg<D>;
  if (cudaFuncSetAttribute(pairs_bwd_tc_v_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM_BYTES) != cudaSuccess) return -1;
  int nitems = p.B * p.Z;
  // persistent CTAs: as many as are resident at once.  TMEM (not visible to the occupancy API, which also under-reports
  // kernels with > 48 KB of dynamic shared memory: it answered 1 for d = 32 and halved the grid) allows 512 / TMEM_COLS
  const int occ = D == 32 ? 512 / C::TMEM_COLS : 1;
  int nsm = 148;
  { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev); }
  const int ctas = occ * nsm;
  int grid = nitems < ctas ? nitems : ctas;
  pairs_bwd_tc_v_kernel<D><<<grid, C::NT, C::SMEM_BYTES, st>>>(p);
  return 1;
}

}  // namespace

int enf_launch_pairs_bwd_tc_v(cudaStream_t st, int d, const EnfPairTcBwdParams& p) {
  if (d == 32) return launch_v<32>(st, p);
  if (d == 128) return launch_v<128>(st, p);
  if (d == 64) return launch_v<64>(st, p);
  return -1;
}
