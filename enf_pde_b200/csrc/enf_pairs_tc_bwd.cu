// Fused (query, latent)-pair BACKWARD on the tensor cores (EnfPrecision::ENF_PREC_BF16, d = 128).
//
// Three kernels, all (field, latent)-major (a CTA owns one latent (b, z) at a time and walks that field's query tiles of
// 128 rows), so per-latent operands load once, per-latent gradients reduce on chip, and weight-gradient accumulators
// live in TMEM:
//
//   A  (this file) value path, top: stream the `that` operand tiles the forward stashed -> m_h -> n_h,
//                          softmax backward (ds), LayerNorm/gelu backward -> dm_h,
//                          wgrad dW3[b,z,h] += that^T dm_h (TMEM), dgrad dthat = sum_h dm_h W3_h^T (TMEM),
//                          out: dthat (fp16), ds, dW3, db3.
//   B  (enf_pairs_tc_bwd_v.cu) value path, bottom: gamma_v -> h1v -> tpre/that; dtpre = LNbwd(dthat) gelu'(tpre);
//                          dW', dW1_v, biases; d gamma_v -> du_v.
//   C  (enf_pairs_tc_bwd_q.cu) query path: gamma_q -> h1q; dzq = scale sum_h ds_h U_h [h1q>0]; dU, dkappa, dW1_q;
//                          d gamma_q -> du; window / invariant backward -> dLam record, dsigma.
//
// TMEM (512 columns) is what forces the split: the five weight-gradient accumulators of the chain need 640
// columns.  Gradient operands are fp16, so all cotangents are pre-scaled by a power of two `gs` that brings
// max|dnbar| to 16; accumulators are multiplied by 1/gs when they are flushed.
#include "enf_pairs_tc_common.cuh"

namespace {

using namespace tcp;

template <int D, int H> struct BwdCfg {
  static constexpr int NQ = D / 32;
  static constexpr int NT = ROWS * NQ;
  static constexpr uint32_t WIMG = wimg_bytes<D>();
  static constexpr uint32_t WBLK = D * 128;
  static constexpr uint32_t ABLK = ROWS * 128;
  static constexpr uint32_t ATILE = atile_bytes<D>();
  static constexpr int HD = D / 2;
  static_assert(H <= 2 || D == 32, "three heads in one kernel A: num_hidden = 32 only; more run as head groups");
};

__device__ __forceinline__ void load_scale(const float* gmax, float& gs, float& inv_gs) {
  float m = *gmax;
  int e = 0;
  if (m > 0.f && isfinite(m)) { frexpf(m, &e); }       // m = f * 2^e, f in [0.5, 1)
  gs = (m > 0.f && isfinite(m)) ? ldexpf(1.f, 4 - e) : 1.f;
  inv_gs = 1.f / gs;
}

// Prep, pass 1: gmax = max |dnbar|
__global__ void __launch_bounds__(256) bwd_prep_max_kernel(const float4* __restrict__ dnbar, int64_t n4, float* gmax) {
  float mx = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 a = __ldg(dnbar + i);
    mx = fmaxf(fmaxf(fmaxf(mx, fabsf(a.x)), fabsf(a.y)), fmaxf(fabsf(a.z), fabsf(a.w)));
  }
  mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<int*>(gmax), __float_as_int(mx));     // non-negative floats order as ints
}
// Prep, pass 2: dnb16 = fp16(gs * dnbar) in the order kernel A loads it (a warp's 16-byte loads are contiguous), and
// Dg[b,c,h] = dnb16 . nbar / gs -- from the ROUNDED cotangent, so that sum_z ds_z = 0 holds exactly as in the forward.
// One thread per (b, c, h, column quarter); rows beyond C are written as zeros.
template <int D>
__global__ void __launch_bounds__(256) bwd_prep_pack_kernel(const float* __restrict__ dnbar, const float* __restrict__ nbar, int B,
                                                            int C, int H, const float* __restrict__ gmax, uint4* __restrict__ dnb16,
                                                            float* __restrict__ Dg) {
  constexpr int NQ = D / 32;
  const int ntiles = (C + 127) / 128;
  float gs, inv_gs;
  load_scale(gmax, gs, inv_gs);
  const int64_t total = (int64_t)B * ntiles * H * NQ * 128;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int row = (int)(t % 128);
    int64_t r = t / 128;
    const int cq = (int)(r % NQ); r /= NQ;
    const int h = (int)(r % H); r /= H;
    const int ct = (int)(r % ntiles);
    const int b = (int)(r / ntiles);
    const int c = ct * 128 + row;
    uint4* dst = dnb16 + ((((int64_t)b * ntiles + ct) * H + h) * NQ + cq) * 4 * 128 + row;       // + q * 128
    float part = 0.f;
    if (c < C) {
      const float4* s4 = reinterpret_cast<const float4*>(dnbar + (((int64_t)b * C + c) * H + h) * D + cq * 32);
      const float4* n4 = reinterpret_cast<const float4*>(nbar + (((int64_t)b * C + c) * H + h) * D + cq * 32);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 a0 = __ldg(s4 + 2 * q), a1 = __ldg(s4 + 2 * q + 1), m0 = __ldg(n4 + 2 * q), m1 = __ldg(n4 + 2 * q + 1);
        const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w}, mv[8] = {m0.x, m0.y, m0.z, m0.w, m1.x, m1.y, m1.z, m1.w};
        uint4 u;
        __half2* h2 = reinterpret_cast<__half2*>(&u);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          h2[k] = __floats2half2_rn(av[2 * k] * gs, av[2 * k + 1] * gs);
          const float2 back = __half22float2(h2[k]);
          part = fmaf(back.x, mv[2 * k], part); part = fmaf(back.y, mv[2 * k + 1], part);
        }
        dst[q * 128] = u;
      }
    } else {
#pragma unroll
      for (int q = 0; q < 4; ++q) dst[q * 128] = make_uint4(0u, 0u, 0u, 0u);
    }
    if (c < C) atomicAdd(Dg + ((int64_t)b * C + c) * H + h, part * inv_gs);
  }
}

// =================================================================================================
// kernel A
// =================================================================================================
// The forward stashed the fp16 operand tile of `that` for every (field, latent, query tile); A streams those tiles
// back with the bulk-copy engine (double buffered) instead of recomputing gamma_v -> h1v -> that, so a tile costs
//     G4_h   m_h = that W3_h                       (one per head; the next tile's first one is issued a tile ahead)
//     E_h    n_h, softmax backward (ds), LayerNorm / gelu backward -> dm_h (fp16 tile, one buffer per head)
//     wgrad  dW3_h += that^T dm_h (TMEM, CTA lifetime)      dgrad  dthat (+)= dm_h W3_h^T
// TMEM: two working regions + H weight-gradient accumulators.  The regions swap roles every tile: the dgrad lands in
// the region the first head's epilogue has already consumed, the region freed by the last head's epilogue receives
// the NEXT tile's first G4, so only the last head's dgrad is ever waited for.
template <int D, int H> struct ACfg {
  using B = BwdCfg<D, H>;
  static constexpr uint32_t OFF_W3 = 0;                              // [H] W3 images
  static constexpr uint32_t OFF_T = H * B::WIMG;                     // [2] that tiles
  static constexpr uint32_t OFF_DM = OFF_T + 2 * B::ATILE;           // [H] dm tiles
  static constexpr uint32_t OFF_F = OFF_DM + H * B::ATILE;
  static constexpr int F_TOTAL = H * D /*b3*/ + 2 * B::NQ * ROWS * 4 /*exchange*/ + H * D /*db3*/ + 2 * 3 * ROWS * H /*row scalars*/;
  static constexpr uint32_t SMEM_BYTES = OFF_F + F_TOTAL * 4 + 128 + 1024;
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
};

// Warp roles: all 16 warps run the epilogues (thread layout of enf_pairs_tc_common.cuh) and never block on each other:
// when their part of an operand tile is written they ARRIVE on a named barrier the issuing warp SYNCs on, and go on with
// whatever does not need that MMA.
constexpr int kABarHead = 5;      // + h (h < 3): dm_h tile written              (named barriers 1..4 belong to row_exchange)
constexpr int kABarDth = 8;       // dthat of the tile has been read out of TMEM
using tc::named_arrive;
using tc::named_sync;

// Warp 0 issues (bulk copies, tcgen05.mma, commits) between its own epilogue phases.
// G (head group): the kernel runs heads h0 .. h0 + H - 1 of a description with HT heads in all (one launch per group, see
// launch_main_groups); every per-head tensor keeps its full-HT layout.  dthat = sum over ALL heads: a group with h0 > 0 adds its
// part to the one the previous groups stored (fp32 add of the stored fp16 value, then one more rounding).  G = false: HT = H,
// h0 = 0, the arguments are unused.
template <int D, int H, bool G>
__global__ void __launch_bounds__(BwdCfg<D, H>::NT, D <= 64 ? 2 : 1) pairs_bwd_tc_a_kernel(EnfPairTcBwdParams P, int h0_arg, int HT_arg) {
  using C = BwdCfg<D, H>;
  using A = ACfg<D, H>;
  const int HT = G ? HT_arg : H, h0 = G ? h0_arg : 0;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);   // 1024-aligned; pointer stays in the shared address space (LDS/STS, not generic LD/ST)
  uint8_t* sW3 = base + A::OFF_W3;
  uint8_t* sT = base + A::OFF_T;
  uint8_t* sDm = base + A::OFF_DM;
  float* f = reinterpret_cast<float*>(base + A::OFF_F);
  float* s_b3 = f; f += H * D;
  float* s_exch = f; f += 2 * C::NQ * ROWS * 4;
  float* s_db3 = f; f += H * D;
  float* s_rs = f; f += 2 * 3 * ROWS * H;             // [2 tiles][logit | lse | Dg][ROWS][H], filled one tile ahead by cp.async
  uint64_t* bars = reinterpret_cast<uint64_t*>(f);
  uint64_t *bar_w = bars, *bar_t = bars + 1 /*[2]*/, *bar_g4 = bars + 3 /*[3]*/, *bar_d = bars + 6, *bar_gb = bars + 7;
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bars + 8);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int lq = warp & 3, cq = warp >> 2;
  const int row = lq * 32 + lane, col0 = cq * 32;
  const int64_t bz = blockIdx.x;
  const int b = (int)(bz / P.Z), z = (int)(bz % P.Z);
  const int ntiles = (P.C + ROWS - 1) / ROWS;
  const uint8_t* timg = P.that_img + (size_t)bz * ntiles * C::ATILE;

  if (tid == 0) {
    for (int i = 0; i < 8; ++i) tc::mbar_init(bars + i, 1);
    tc::mbar_fence_init();
  }
  // two working regions (three with three heads: the third head's m has a region of its own) + H weight-gradient
  // accumulators; at d <= 64 that is at most half of TMEM (and of shared memory, and 128 registers per thread for <= 256
  // threads): two CTAs per SM, each filling the other's MMA / barrier waits
  constexpr int kWork = H == 3 ? 3 : 2;
  constexpr int kTmemNeed = (kWork + H) * D;
  constexpr int kTmemCols = kTmemNeed <= 128 ? 128 : kTmemNeed <= 256 ? 256 : 512;
  if (warp == 0) tc::tmem_alloc<kTmemCols>(s_tmem);
  for (int e = tid; e < H * D; e += C::NT) { s_b3[e] = P.b3[(G ? (bz * HT + h0) * D : bz * H * D) + e]; s_db3[e] = 0.f; }
  float gs, inv_gs;
  load_scale(P.gmax, gs, inv_gs);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tm = *s_tmem;
  const uint32_t tW3 = tm + kWork * D, tR2 = tm + 2 * D;      // tR2: working region of the third head (H = 3)
  const uint32_t lane_off = (uint32_t)(lq * 32) << 16;
  const uint32_t my_t = lane_off + col0;
  const uint32_t aW3 = tc::smem_u32(sW3), aT = tc::smem_u32(sT), aDm = tc::smem_u32(sDm);

  // ---- what the issuing lane does at the three issue points of a tile ------------------------------------------------------
  auto issue_prologue = [&]() {
    tc::mbar_expect_tx(bar_w, H * C::WIMG);
    for (int h = 0; h < H; ++h) tc::bulk_g2s(sW3 + h * C::WIMG, P.img_W3 + (G ? bz * HT + h0 + h : bz * H + h) * C::WIMG, C::WIMG, bar_w);
    tc::mbar_expect_tx(&bar_t[0], C::ATILE);
    tc::bulk_g2s(sT, timg, C::ATILE, &bar_t[0]);
    tc::mbar_wait(bar_w, 0);
    tc::mbar_wait(&bar_t[0], 0);
    tc::tc_fence_after();
    issue_gemm<D>(tm, aT, aW3, C::ABLK, C::WBLK);               // m_0 of tile 0 -> region 0
    tc::mma_commit(&bar_g4[0]);
  };
  auto issue_top = [&](int ct) {                      // tS (= the previous tile's dgrad region) has been read by every epilogue thread
    const int e = ct & 1;
    tc::tc_fence_after();
    if (H > 1) {
      issue_gemm<D>(tm + (e ^ 1) * D, aT + e * C::ATILE, aW3 + C::WIMG, C::ABLK, C::WBLK);
      tc::mma_commit(&bar_g4[1]);
    }
    if (H > 2) {                                      // every head's epilogue of the previous tile is behind the barrier too
      issue_gemm<D>(tR2, aT + e * C::ATILE, aW3 + 2 * C::WIMG, C::ABLK, C::WBLK);
      tc::mma_commit(&bar_g4[2]);
    }
    if (ct + 1 < ntiles) {                            // next that tile -> the other buffer, once the previous tile's wgrad has read it
      if (ct > 0) tc::mbar_wait(bar_gb, (ct - 1) & 1);
      tc::mbar_expect_tx(&bar_t[e ^ 1], C::ATILE);
      tc::bulk_g2s(sT + (e ^ 1) * C::ATILE, timg + (size_t)(ct + 1) * C::ATILE, C::ATILE, &bar_t[e ^ 1]);
    }
  };
  auto issue_head = [&](int ct, int h) {              // dm_h is in shared memory
    const int e = ct & 1;
    const uint32_t tF = tm + e * D, tS = tm + (e ^ 1) * D;
    const uint32_t aTc = aT + e * C::ATILE;
    tc::tc_fence_after();
    const uint32_t aDh = aDm + h * C::ATILE, aWh = aW3 + h * C::WIMG;
    if (h + 1 < H) {
      issue_wgrad<D>(tW3 + h * D, aTc, aDh, C::ABLK, ct > 0);
      issue_dgrad<D>(tF, aDh, aWh, C::ABLK, C::WBLK, h > 0);
    } else {
      issue_dgrad<D>(tF, aDh, aWh, C::ABLK, C::WBLK, h > 0);
      tc::mma_commit(bar_d);
      issue_wgrad<D>(tW3 + h * D, aTc, aDh, C::ABLK, ct > 0);
      tc::mma_commit(bar_gb);
      if (ct + 1 < ntiles) {                          // tS is consumed: the next tile's first G4 goes there now
        tc::mbar_wait(&bar_t[e ^ 1], ((ct + 1) >> 1) & 1);
        tc::tc_fence_after();
        issue_gemm<D>(tS, aT + (e ^ 1) * C::ATILE, aW3, C::ABLK, C::WBLK);
        tc::mma_commit(&bar_g4[0]);
      }
    }
  };

  int xw = 0;
  // per-row scalars of tile `ct` (logits, log-sum-exp, Dg of my row, all heads) -> shared, without passing through registers
  auto prefetch_rows = [&](int ct) {
    const int c = ct * ROWS + row;
    if (cq == 0 && c < P.C) {
      const int64_t q = (int64_t)b * P.C + c;
      float* dst = s_rs + (ct & 1) * 3 * ROWS * H + row * H;
      if (H == 3 || G) {   // 12 bytes is not a cp.async size; a group of two at an odd head (or of HT = 3) is only 4-byte aligned
#pragma unroll
        for (int h = 0; h < H; ++h) {
          tc::cp_async<4>(dst + h, P.slog + (bz * P.C + c) * HT + h0 + h);
          tc::cp_async<4>(dst + ROWS * H + h, P.lse + q * HT + h0 + h);
          tc::cp_async<4>(dst + 2 * ROWS * H + h, P.Dg + q * HT + h0 + h);
        }
      } else {
        constexpr int kB = 4 * (H == 3 ? 1 : H);
        tc::cp_async<kB>(dst, P.slog + (bz * P.C + c) * H);
        tc::cp_async<kB>(dst + ROWS * H, P.lse + q * H);
        tc::cp_async<kB>(dst + 2 * ROWS * H, P.Dg + q * H);
      }
    }
  };
  if (warp == 0) {
    if (tc::elect_one()) issue_prologue();
    __syncwarp();
  }
  prefetch_rows(0);
  uint4 dnq[4];                                      // my 32 columns of the scaled fp16 cotangent of nbar, (tile, head) about to be processed
  auto load_dnb = [&](int ct, int h) {
    const uint4* src = P.dnb16 + ((((int64_t)b * ntiles + ct) * HT + h0 + h) * C::NQ + cq) * 4 * ROWS + row;
#pragma unroll
    for (int q = 0; q < 4; ++q) dnq[q] = __ldg(src + q * ROWS);       // a warp reads 512 contiguous bytes per instruction
  };
  load_dnb(0, 0);

  for (int ct = 0; ct < ntiles; ++ct) {
    const uint32_t par = ct & 1;
    const int e = ct & 1;                            // region roles of this tile: first = region e, other = region e ^ 1
    const uint32_t tF = tm + e * D, tS = tm + (e ^ 1) * D;
    const int c0 = ct * ROWS;
    const bool valid = c0 + row < P.C;
    if (warp == 0) {                                 // warp 0 doubles as the issuer
      if (ct > 0) named_sync(kABarDth, C::NT);
      if (tc::elect_one()) issue_top(ct);
      __syncwarp();
    }
    tc::cp_async_wait_all();                         // this tile's row scalars (issued a tile ago by the cq == 0 thread of the row);
                                                     // the row's other threads read them after the row_exchange barrier below
    if (ct + 1 < ntiles) prefetch_rows(ct + 1);
    float v[32];
#pragma unroll
    for (int h = 0; h < H; ++h) {
      tc::mbar_wait(&bar_g4[h], par);
      tc::tc_fence_after();
      tc::tmem_ld32((h == 0 ? tF : h == 1 ? tS : tR2) + my_t, v);
      tc::tmem_ld_wait();
      // one pass, one exchange: with g = gelu(m), n = (g - mu) rstd the row sums the LayerNorm backward needs are
      //   sum_j dnb_j n_j = rstd (sum dnb g - mu sum dnb)   and   sum_j dnb_j
      uint32_t dgh[16];                              // gelu', packed to fp16 inside the pass (dm is rounded to fp16 for the MMAs anyway)
      uint32_t gh[16];                               // g, packed to fp16 once the row sums have seen it in fp32 (it only re-enters
                                                     // through the small LayerNorm projection term of dm): 16 registers instead of 32
      float st[4];
      {
        float st01[2];
        gelu_rowsums32_stash(v, s_b3 + h * D + col0, dgh, st01);
        st[0] = st01[0]; st[1] = st01[1];
      }
      // the cotangent rows were requested one phase ago; touching them only now keeps their L2 latency off the gelu pass
      {
        float2 s2 = tc::splat2(0.f), s3 = tc::splat2(0.f);
#pragma unroll
        for (int j4 = 0; j4 < 32; j4 += 4) {
          const __half2* h2 = reinterpret_cast<const __half2*>(&dnq[j4 >> 3]) + ((j4 & 4) >> 1);     // dnb[j4 .. j4 + 3], packed
          const float2 d01 = __half22float2(h2[0]), d23 = __half22float2(h2[1]);
          s2 = tc::fma2(d01, tc::ld2(v + j4), s2); s3 = tc::add2(s3, d01);
          s2 = tc::fma2(d23, tc::ld2(v + j4 + 2), s2); s3 = tc::add2(s3, d23);
          gh[j4 >> 1] = tc::pack_bf16(v[j4], v[j4 + 1]);
          gh[(j4 >> 1) + 1] = tc::pack_bf16(v[j4 + 2], v[j4 + 3]);
        }
        st[2] = s2.x + s2.y; st[3] = s3.x + s3.y;
      }
      row_exchange<C::NQ, 4>(s_exch, xw, cq, row, lq, st);
      float att = 0.f, Dh = 0.f;
      if (valid) {
        const float* rs = s_rs + e * 3 * ROWS * H + row * H + h;
        att = __expf(rs[0] - rs[ROWS * H]);
        Dh = rs[2 * ROWS * H];
      }
      const float atts = att;                        // dnb16 already carries the scale gs
      const float mu = st[0] * (1.f / D);
      const float rstd = rsqrtf(fmaxf(st[1] * (1.f / D) - mu * mu, 0.f) + 1e-6f);
      const float dd0 = rstd * (st[2] - mu * st[3]), dd1 = st[3];
      const float dsh = atts * (dd0 - Dh * gs);
      const float mean1 = atts * dd1 * (1.f / D), mean2 = atts * dd0 * (1.f / D);
      // dm = rstd (att dnb - mean1 - n mean2) g'   with n = (g - mu) rstd, constants folded
      const float ka = atts * rstd, kc = rstd * (mu * rstd * mean2 - mean1), kb = rstd * rstd * mean2;
      uint8_t* sDh = sDm + h * C::ATILE;
      if (h == 0 && ct > 0) tc::mbar_wait(bar_gb, par ^ 1);      // every MMA of the previous tile is done with the dm tiles
      uint32_t dmh[16];                              // dm as the fp16 operand words the MMAs read; the bias column sums add the same words
#pragma unroll
      for (int c8 = 0; c8 < 32; c8 += 8) {
        const __half2* h2 = reinterpret_cast<const __half2*>(&dnq[c8 >> 3]);
        const __half2* g2 = reinterpret_cast<const __half2*>(&gh[c8 >> 1]);
        const __half2* d2 = reinterpret_cast<const __half2*>(&dgh[c8 >> 1]);
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const float2 dv = __half22float2(h2[t]), gv = __half22float2(g2[t]);
          const float2 dm = tc::mul2(tc::fma2(gv, tc::splat2(-kb), tc::fma2(tc::splat2(ka), dv, tc::splat2(kc))), __half22float2(d2[t]));
          dmh[(c8 >> 1) + t] = tc::pack_bf16(dm.x, dm.y);
        }
        tc::st_row8_words(sDh, C::ABLK, row, col0 + c8, dmh + (c8 >> 1));
      }
      tc::fence_proxy_async();
      tc::tc_fence_before();
      if (warp == 0) {
        named_sync(kABarHead + h, C::NT);
        if (tc::elect_one()) issue_head(ct, h);
        __syncwarp();
      } else {
        named_arrive(kABarHead + h, C::NT);            // warp 0 takes it from here
      }
      // fetch the cotangent rows of the next (tile, head) now, a whole phase ahead of their use
      if (h + 1 < H) load_dnb(ct, h + 1);
      else if (ct + 1 < ntiles) load_dnb(ct + 1, 0);
      {
        float cs = warp_colsum32_h2(dmh, lane);
        atomicAdd(&s_db3[h * D + col0 + lane], cs);
      }
      if (cq == 0 && valid) P.ds[((bz * P.C) + c0 + row) * HT + h0 + h] = dsh;
    }
    // dthat = sum_h dm_h W3_h^T -> global (fp16, scaled)
    tc::mbar_wait(bar_d, par);
    tc::tc_fence_after();
    tc::tmem_ld32(tF + my_t, v);
    tc::tmem_ld_wait();
    tc::tc_fence_before();
    if (ct + 1 < ntiles && warp != 0) named_arrive(kABarDth, C::NT);     // tF may be overwritten by the next tile's second G4
    {                                                // chunked order: a warp stores 512 contiguous bytes per instruction
      uint4* dst = reinterpret_cast<uint4*>(P.dthat) + ((bz * ntiles + ct) * C::NQ + cq) * 4 * ROWS + row;
      if constexpr (G) {
        if (h0 > 0) {                                // the earlier groups' part of dthat
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const uint4 prev = dst[q * ROWS];
            const __half2* p2 = reinterpret_cast<const __half2*>(&prev);
#pragma unroll
            for (int t = 0; t < 4; ++t) tc::st2(v + q * 8 + 2 * t, tc::add2(tc::ld2(v + q * 8 + 2 * t), __half22float2(p2[t])));
          }
        }
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        uint4 u;
        __half2* h2 = reinterpret_cast<__half2*>(&u);
#pragma unroll
        for (int t = 0; t < 4; ++t) h2[t] = __floats2half2_rn(v[q * 8 + 2 * t], v[q * 8 + 2 * t + 1]);
        dst[q * ROWS] = u;
      }
    }
  }
  tc::mbar_wait(bar_gb, (ntiles - 1) & 1);
  tc::tc_fence_after();
  // flush dW3[b,z,h] (lane = input feature, column = output feature) and db3
  __syncthreads();
  tc::tc_fence_after();
  // accumulator row (input feature) of this thread (enf_pairs_tc_common.cuh: wgrad_row)
  const int wrow = wgrad_row<D>(row, lq, lane);
#pragma unroll
  for (int h = 0; h < H; ++h) {
    float w[32];
    tc::tmem_ld32(tW3 + h * D + my_t, w);
    tc::tmem_ld_wait();
    if (wrow >= 0) {
      float* o = P.g_W3 + ((G ? bz * HT + h0 + h : bz * H + h) * D + wrow) * D + col0;
#pragma unroll
      for (int j = 0; j < 32; j += 4)
        *reinterpret_cast<float4*>(o + j) = make_float4(w[j] * inv_gs, w[j + 1] * inv_gs, w[j + 2] * inv_gs, w[j + 3] * inv_gs);
    }
  }
  for (int e = tid; e < H * D; e += C::NT) P.g_b3[(G ? (bz * HT + h0) * D : bz * H * D) + e] = s_db3[e] * inv_gs;
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc<kTmemCols>(tm);
}

template <int D>
int launch_prep(cudaStream_t st, int H, const EnfPairTcBwdParams& p) {
  const int64_t n4 = (int64_t)p.B * p.C * H * D / 4;
  int blocks = (int)((n4 + 255) / 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  bwd_prep_max_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<const float4*>(p.dnbar), n4, const_cast<float*>(p.gmax));
  if (cudaMemsetAsync(p.Dg, 0, (size_t)p.B * p.C * H * sizeof(float), st) != cudaSuccess) return -1;
  bwd_prep_pack_kernel<D><<<148 * 8, 256, 0, st>>>(p.dnbar, p.nbar, p.B, p.C, H, p.gmax, p.dnb16, p.Dg);
  return 2;
}

template <int D, int H, bool G = false>
int launch_a(cudaStream_t st, const EnfPairTcBwdParams& p, int h0 = 0, int HT = H) {
  using C = BwdCfg<D, H>;
  size_t smem_a = ACfg<D, H>::SMEM_BYTES;
  if (cudaFuncSetAttribute(pairs_bwd_tc_a_kernel<D, H, G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_a) != cudaSuccess) return -1;
  const unsigned grid = (unsigned)(p.B * p.Z);
  pairs_bwd_tc_a_kernel<D, H, G><<<grid, C::NT, smem_a, st>>>(p, h0, HT);
  return 1;
}

template <int D, int H>
int launch_main(cudaStream_t st, const EnfPairTcBwdParams& p) {
  if (launch_a<D, H>(st, p) < 0) return -1;
  if (enf_launch_pairs_bwd_tc_v(st, D, p) < 0) return -1;
  if (enf_launch_pairs_bwd_tc_q(st, D, H, p) < 0) return -1;
  return 3;
}

// More heads than kernel A holds in TMEM: one kernel A per group of at most two heads (H = 3: 2 + 1, H = 4: 2 + 2), in head
// order, the later groups adding to dthat; kernel B does not depend on the heads and kernel C runs once with all of them.
template <int D>
int launch_main_groups(cudaStream_t st, int H, const EnfPairTcBwdParams& p) {
  int n = 0;
  for (int h0 = 0; h0 < H; h0 += 2) {
    if ((H - h0 >= 2 ? launch_a<D, 2, true>(st, p, h0, H) : launch_a<D, 1, true>(st, p, h0, H)) < 0) return -1;
    ++n;
  }
  if (enf_launch_pairs_bwd_tc_v(st, D, p) < 0) return -1;
  if (enf_launch_pairs_bwd_tc_q(st, D, H, p) < 0) return -1;
  return n + 2;
}

}  // namespace

bool enf_pairs_bwd_tc_supported(int d, int H) { return (d == 128 || d == 64 || d == 32) && H >= 1 && H <= 4; }

int enf_launch_pairs_bwd_tc_prep(cudaStream_t st, int d, int H, const EnfPairTcBwdParams& p) {
  if (!enf_pairs_bwd_tc_supported(d, H)) return -1;
  if (d == 32) return launch_prep<32>(st, H, p);
  if (d == 128) return launch_prep<128>(st, H, p);
  return launch_prep<64>(st, H, p);
}

int enf_launch_pairs_bwd_tc_main(cudaStream_t st, int d, int H, const EnfPairTcBwdParams& p) {
  if (d == 32 && H == 4) return launch_main_groups<32>(st, H, p);
  if (d == 128 && H > 2) return launch_main_groups<128>(st, H, p);
  if (d == 64 && H > 2) return launch_main_groups<64>(st, H, p);
  if (d == 32 && H == 3) return launch_main<32, 3>(st, p);
  if (d == 32 && H == 2) return launch_main<32, 2>(st, p);
  if (d == 32 && H == 1) return launch_main<32, 1>(st, p);
  if (d == 128 && H == 2) return launch_main<128, 2>(st, p);
  if (d == 128 && H == 1) return launch_main<128, 1>(st, p);
  if (d == 64 && H == 2) return launch_main<64, 2>(st, p);
  if (d == 64 && H == 1) return launch_main<64, 1>(st, p);
  return -1;
}
