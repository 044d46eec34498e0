// Fused (query, latent)-pair FORWARD kernel on the 5th-gen tensor cores (EnfPrecision::ENF_PREC_BF16).
//
// One CTA owns 128 coordinate queries of one field (= the 128 TMEM lanes / UMMA M) and loops over the
// field's Z latents.  Per latent the chain of equivariant_cross_attention.py:86-144 runs as
//     E0q  gamma_q -> smem A0 (fp16, 128B swizzle)        GEMM1  A0 x W1_q      -> TMEM T1
//     E0v  gamma_v -> smem A1                             GEMM2  A1 x W1_v      -> TMEM T0
//     E1   T1: relu, dot with folded U[z,h] -> logits s ; online-softmax statistics
//     E2   T0: relu -> A0                                 GEMM3  A0 x W'        -> T0
//     E3   T0: gelu, LayerNorm -> A1                      GEMM4h A1 x W3[z,h]   -> T0 / T1
//     E4h  Th: gelu, LayerNorm, acc_h = acc_h corr + p n                             (TMEM, tcgen05.ld / st)
// with tcgen05.mma (kind::f16, fp16 operands, fp32 accumulators in TMEM) issued by one thread, weights
// resident in shared memory as pre-swizzled images, the per-latent W3 images streamed by the bulk-copy
// (TMA) engine, tcgen05.ld feeding the elementwise epilogues, D/32 threads per query row.  TMEM holds the two working
// regions T0 / T1 (T0 also receives the next latent's RFF phases once E4_0 has read it) and the H softmax-weighted
// accumulators (H x d fp32 per row): keeping those out of the register file is what lets ptxas keep several dependent
// chains of the epilogues in flight.  The epilogues use packed fp32 pairs (FFMA2 / FMUL2 / FADD2) and evaluate the cosines
// of the RFF phases on the FMA pipe (the XU pipe only sees the sines and the tanh of the gelus).  Per pair, HBM only sees
// what is saved for the backward: the logits, the fp16 operand tile of `that` (bulk-stored straight from shared memory) and
// gelu'(tpre) / rstd of that layer for backward kernel B (staged in the W3 stage buffer, one bulk store per latent).  MMA
// and epilogues overlap where the chain allows it (GEMM1 | E0v, GEMM2 | E1, GEMM3 | softmax update, GEMM4_1 | E4_0).
#include "enf_pairs_tc_common.cuh"

namespace {

using namespace tcp;

template <int D, int H> struct TcCfg {
  static constexpr int NQ = D / 32;                    // threads per query row (32 columns each)
  static constexpr int NT = ROWS * NQ;                 // threads per CTA
  static constexpr uint32_t WIMG = wimg_bytes<D>();    // bytes of one weight image
  static constexpr uint32_t WBLK = D * 128;            // bytes of one 64-feature block of a weight image
  static constexpr uint32_t ABLK = ROWS * 128;         // bytes of one 64-feature block of an activation tile
  static constexpr uint32_t ATILE = atile_bytes<D>();
  static constexpr uint32_t DTILE = ROWS * D * 2;      // bytes of one tile of the gelu' stash (fp16, chunked order)
  // d = 32: the images are small, so ALL heads' W3[z,h] are staged together one latent ahead (d >= 64 streams W3[z,1] into the
  // A0 tile once GEMM3 has released it), and with H = 3 the third head's GEMM4 reuses T0 after E4_0, which moves the next
  // latent's RFF phases to a region of their own
  static constexpr bool kStageAll = D == 32;
  static constexpr uint32_t SBYTES = kStageAll ? H * WIMG : WIMG;
  static constexpr bool kOwnPhaseRegion = H == 3;
  static constexpr int TMEM_NEED = (2 + H) * D + (kOwnPhaseRegion ? D : 0);
  static constexpr int TMEM_COLS = TMEM_NEED <= 128 ? 128 : TMEM_NEED <= 256 ? 256 : 512;   // T0 (also the RFF phases of the next latent) | T1 | H softmax accumulators
  // byte offsets inside the 1024-aligned dynamic shared memory
  static constexpr uint32_t OFF_W = 0;                 // W1_q, W1_v, W' images
  static constexpr uint32_t OFF_S = 3 * WIMG;          // W3[z,0] stage (d = 32: W3[z,0..H-1])
  static constexpr uint32_t OFF_A0 = OFF_S + SBYTES;
  static constexpr uint32_t OFF_A1 = OFF_A0 + ATILE;
  static constexpr uint32_t OFF_U = OFF_A1 + ATILE;    // projection operand: invariants of the 128 rows (2 atoms)
  static constexpr uint32_t OFF_OM = OFF_U + 2 * kProjAtom;   // projection operand: [Omega_q | Omega_v] (D / 64 atoms)
  // staging of the backward's stash rstd * gelu' (one activation tile): the W3 stage buffer where that is large enough (d = 128)
  static constexpr uint32_t OFF_G = OFF_OM + nblk<D>() * kProjAtom;
  static constexpr uint32_t OFF_F = OFF_G + (WIMG >= ATILE ? 0 : ATILE);    // float arrays start here
  // float arrays (counts)
  // per-latent vectors are double buffered (cp.async prefetch of the next latent): [2] x { Lam 64 | U H*D | b3 H*D | kappa, sigma 8 }
  static constexpr int F_LAT = 64 + 2 * H * D + 8;
  static constexpr int F_WIN = 2 * ROWS, F_BIAS = 3 * D, F_EXCH = NQ * ROWS * 2 + NQ * ROWS * (H > 2 ? H : 2);
  static_assert(H <= 2 || D == 32, "three heads in one kernel: num_hidden = 32 only (TMEM: T0 | T1 | H accumulators | phases); more run as head groups");
  static_assert(H <= 3, "the logit partials [NQ][ROWS][H] share exchange buffer 1");
  static constexpr int F_TOTAL = 2 * F_LAT + F_WIN + F_BIAS + F_EXCH;
  static constexpr uint32_t SMEM_BYTES = OFF_F + F_TOTAL * 4 + 128 /*barriers*/ + 1024 /*alignment slack*/;
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
};

// G (head group): the kernel runs heads h0 .. h0 + H - 1 of a description with HT heads in all (one launch per group, see
// enf_launch_pairs_fwd_tc); every per-head tensor keeps its full-HT layout.  G = false: HT = H, h0 = 0, the arguments are unused.
template <int D, int H, bool G>
__global__ void __launch_bounds__(TcCfg<D, H>::NT, D <= 64 ? 2 : 1) pairs_fwd_tc_kernel(EnfPairTcParams P, int h0_arg, int HT_arg) {
  using C = TcCfg<D, H>;
  const int HT = G ? HT_arg : H, h0 = G ? h0_arg : 0;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);   // 1024-aligned; pointer stays in the shared address space (LDS/STS, not generic LD/ST)
  uint8_t* sW = base + C::OFF_W;
  uint8_t* sS = base + C::OFF_S;
  uint8_t* sA0 = base + C::OFF_A0;
  uint8_t* sA1 = base + C::OFF_A1;
  uint8_t* sU = base + C::OFF_U;
  uint8_t* sOm = base + C::OFF_OM;
  uint8_t* sG = C::WIMG >= C::ATILE ? sS : base + C::OFF_G;
  float* f = reinterpret_cast<float*>(base + C::OFF_F);
  float* s_lat = f; f += 2 * C::F_LAT;        // [2] per-latent vectors of this and the next latent
  float* s_win = f; f += C::F_WIN;            // [2][ROWS]: window values of this and the next latent
  float* s_bias = f; f += C::F_BIAS;          // b1q | b1v | bp
  float* s_exch = f; f += C::F_EXCH;          // two [NQ][ROWS][2] exchange buffers: 0 = E3 and E4_1, 1 = E4_0
  float* s_spart = s_exch + C::NQ * ROWS * 2; // [NQ][ROWS][H] logit partials live in buffer 1 between E1 and the softmax statistics
  uint64_t* bars = reinterpret_cast<uint64_t*>(f);
  uint64_t* bar_w = bars + 0;
  uint64_t* bar_g1 = bars + 1;
  uint64_t* bar_g2 = bars + 2;
  uint64_t* bar_g3 = bars + 3;
  uint64_t* bar_g4 = bars + 4;                // [3]
  uint64_t* bar_w3 = bars + 7;                // [2]
  uint64_t* bar_p = bars + 9;                 // RFF phases of the next latent are in TMEM
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bars + 10);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int lq = warp & 3, cq = warp >> 2;
  const int row = lq * 32 + lane, col0 = cq * 32;
  const int b = blockIdx.y, c0 = blockIdx.x * ROWS;
  const bool row_valid = c0 + row < P.C;
  const float scale = rsqrtf((float)D);
  constexpr int HD = D / 2;

  if (tid == 0) {
    for (int i = 0; i < 10; ++i) tc::mbar_init(bars + i, 1);
    tc::mbar_fence_init();
  }
  if (warp == 0) tc::tmem_alloc<C::TMEM_COLS>(s_tmem);
  // per-CTA constants
  for (int e = tid; e < D; e += C::NT) { s_bias[e] = P.q_b1[e]; s_bias[D + e] = P.v_b1[e]; s_bias[2 * D + e] = P.bp[e]; }
  // per-latent vectors of latent z -> buffer z & 1, without passing through registers (16-byte cp.async each)
  auto prefetch_latent = [&](int z) {
    const int64_t q = (int64_t)b * P.Z + z;
    float* dst = s_lat + (z & 1) * C::F_LAT;
    constexpr int NU = H * D / 4;
    const int64_t qh = G ? q * HT + h0 : q * H;        // this group's first head of latent q
    if (tid < NU) tc::cp_async<16>(dst + 64 + 4 * tid, P.U + qh * D + 4 * tid);
    else if (tid < 2 * NU) tc::cp_async<16>(dst + 64 + H * D + 4 * (tid - NU), P.b3 + qh * D + 4 * (tid - NU));
    else if (tid < 2 * NU + ENF_LAM_SIZE / 4) tc::cp_async<16>(dst + 4 * (tid - 2 * NU), P.lam + q * ENF_LAM_SIZE + 4 * (tid - 2 * NU));
    else if (tid == 2 * NU + ENF_LAM_SIZE / 4) {
      if (H == 3 || G) {     // 12 bytes is not a cp.async size (and q * 12 bytes, or a group at an odd head, is only 4-byte aligned)
#pragma unroll
        for (int h = 0; h < H; ++h) tc::cp_async<4>(dst + 64 + 2 * H * D + h, P.kappa + qh + h);
      } else {
        tc::cp_async<4 * (H == 3 ? 1 : H)>(dst + 64 + 2 * H * D, P.kappa + q * H);
      }
    }
    else if (tid == 2 * NU + ENF_LAM_SIZE / 4 + 1 && P.sigma) tc::cp_async<4>(dst + 64 + 2 * H * D + 4, P.sigma + q);
  };
  prefetch_latent(0);
  tc::cp_async_wait_all();
  proj_zero(sU, 2, tid, C::NT);
  proj_zero(sOm, nblk<D>(), tid, C::NT);
  // every thread keeps its row's query features in registers for the whole kernel (the NQ threads of a row share the
  // invariant rows of the next latent between them)
  float xi_r[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) xi_r[k] = 0.f;
  if (row_valid) {
    const float4* src = reinterpret_cast<const float4*>(P.xi + (int64_t)b * P.xi_bs + (int64_t)(c0 + row) * 8);
    float4 a = __ldg(src), c = __ldg(src + 1);
    xi_r[0] = a.x; xi_r[1] = a.y; xi_r[2] = a.z; xi_r[3] = a.w; xi_r[4] = c.x; xi_r[5] = c.y; xi_r[6] = c.z; xi_r[7] = c.w;
  }
  // invariants of latent `buf`'s record -> projection operand: thread cq of a row computes rows cq and cq + NQ, the last
  // thread of the row also the window value
  auto write_invariants = [&](const float* lat, int wbuf) {
#pragma unroll
    for (int k = 0; k < (6 + C::NQ - 1) / C::NQ; ++k) {
      const int i = cq + k * C::NQ;
      if (i < P.rec.I && i < 6) proj_store_pair(sU, i, row, record_row(P.rec, lat, xi_r, i), true);
    }
    if (cq == C::NQ - 1) {
      float u0, u1, w, c;
      record_window_rows(P.rec, lat, xi_r, u0, u1);
      record_window<true>(P.rec, lat, xi_r, P.sigma ? lat[64 + 2 * H * D + 4] : 1.f, u0, u1, w, c);
      s_win[wbuf * ROWS + row] = w;
    }
  };
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tm = *s_tmem;
  // T0 doubles as the landing zone of the next latent's RFF phases (issued once E4_0 has read it), which leaves H x D columns
  // for the softmax-weighted accumulators: they live in TMEM (tcgen05.ld / st once per latent and head), not in 64 registers
  // per thread, so that the epilogues have registers for more than one dependent chain in flight.
  const uint32_t t0 = tm, t1 = tm + D, tacc = tm + 2 * D, tp = C::kOwnPhaseRegion ? tm + (2 + H) * D : tm;
  const uint32_t lane_off = (uint32_t)(lq * 32) << 16;
  const uint32_t my_t = lane_off + col0;      // lane-quadrant / column offset of this warp

  if (tid == 0) {
    tc::mbar_expect_tx(bar_w, 3 * C::WIMG);
    tc::bulk_g2s(sW, P.img_q_w1, C::WIMG, bar_w);
    tc::bulk_g2s(sW + C::WIMG, P.img_v_w1, C::WIMG, bar_w);
    tc::bulk_g2s(sW + 2 * C::WIMG, P.img_Wp, C::WIMG, bar_w);
    tc::mbar_expect_tx(&bar_w3[0], C::SBYTES);
    tc::bulk_g2s(sS, P.img_W3 + ((int64_t)b * P.Z * HT + h0) * C::WIMG, C::SBYTES, &bar_w3[0]);
  }
  const uint32_t aA0 = tc::smem_u32(sA0), aA1 = tc::smem_u32(sA1), aS = tc::smem_u32(sS), aW = tc::smem_u32(sW);
  const uint32_t aU = tc::smem_u32(sU), aOm = tc::smem_u32(sOm);

  // Omega image [Omega_q | Omega_v]; invariants of latent 0; phases of latent 0
  proj_build_omega(sOm, 0, P.q_omega, P.rec.I, HD, tid, C::NT);
  proj_build_omega(sOm, HD, P.v_omega, P.rec.I, HD, tid, C::NT);
  __syncthreads();                             // latent 0's vectors are visible
  write_invariants(s_lat, 0);
  tc::fence_proxy_async();
  __syncthreads();
  if (tid == 0) {
    tc::tc_fence_after();
    issue_proj(tp, aU, aOm, D);
    tc::mma_commit(bar_p);
  }

  int xw = 0;                                  // which exchange buffer is next
  float m_run[H], l_run[H];
  {
    float zero[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) zero[j] = 0.f;
#pragma unroll
    for (int h = 0; h < H; ++h) {
      m_run[h] = -INFINITY; l_run[h] = 0.f;
      tc::tmem_st32(tacc + h * D + my_t, zero);
    }
    tc::tmem_st_wait();
  }

  for (int z = 0; z < P.Z; ++z) {
    const uint32_t par = z & 1;
    const int64_t bz = (int64_t)b * P.Z + z;
    const bool more = z + 1 < P.Z;
    // ---- (a) RFF phases of this latent (its invariants were written during the previous latent's E4); prefetch of the
    //          next latent's vectors; gamma_q, gamma_v from the phases
    if (more) prefetch_latent(z + 1);
    const float* s_lam_next = s_lat + (par ^ 1) * C::F_LAT;
    const float* s_uz = s_lat + par * C::F_LAT + 64;
    const float* s_b3 = s_uz + H * D;
    const float* s_kap = s_b3 + H * D;
    tc::mbar_wait(bar_p, par);
    tc::tc_fence_after();
    // gamma_q first: GEMM1 is issued as soon as its operand is complete (named barrier 7: warp 0 syncs, the others arrive)
    // and runs in the shadow of the gamma_v pass
    rff_from_proj<D, false>(tp + lane_off + 16 * cq, sA0, nullptr, C::ABLK, row, 16 * cq);
    tc::fence_proxy_async();
    if (warp == 0) {
      tc::named_sync(7, C::NT);
      if (tid == 0) {
        if (z == 0) tc::mbar_wait(bar_w, 0);
        tc::tc_fence_after();
        issue_gemm<D>(t1, aA0, aW, C::ABLK, C::WBLK);         // T0 still holds the v half of the phases
        tc::mma_commit(bar_g1);
      }
      __syncwarp();
    } else {
      tc::named_arrive(7, C::NT);
    }
    rff_from_proj<D, false>(tp + lane_off + HD + 16 * cq, sA1, nullptr, C::ABLK, row, 16 * cq);
    tc::tc_fence_before();
    tc::fence_proxy_async();
    __syncthreads();
    if (tid == 0) {
      tc::tc_fence_after();
      issue_gemm<D>(t0, aA1, aW + C::WIMG, C::ABLK, C::WBLK);
      tc::mma_commit(bar_g2);
    }
    const float win = s_win[par * ROWS + row];
    // ---- (c) E1: h1q = relu(T0 + b1q); logit partials (overlaps GEMM2) -------------------------------------
    float v[32];
    tc::mbar_wait(bar_g1, par);
    tc::tc_fence_after();
    tc::tmem_ld32(t1 + my_t, v);
    tc::tmem_ld_wait();
    {
      float2 part[H];                          // even / odd columns (packed FFMA2)
#pragma unroll
      for (int h = 0; h < H; ++h) part[h] = tc::splat2(0.f);
#pragma unroll
      for (int j4 = 0; j4 < 32; j4 += 4) {
        const float4 bb = *reinterpret_cast<const float4*>(s_bias + col0 + j4);
        float2 h01 = tc::add2(tc::ld2(v + j4), make_float2(bb.x, bb.y)), h23 = tc::add2(tc::ld2(v + j4 + 2), make_float2(bb.z, bb.w));
        h01.x = fmaxf(h01.x, 0.f); h01.y = fmaxf(h01.y, 0.f); h23.x = fmaxf(h23.x, 0.f); h23.y = fmaxf(h23.y, 0.f);
#pragma unroll
        for (int h = 0; h < H; ++h) {
          const float4 uu = *reinterpret_cast<const float4*>(s_uz + h * D + col0 + j4);
          part[h] = tc::fma2(h01, make_float2(uu.x, uu.y), part[h]);
          part[h] = tc::fma2(h23, make_float2(uu.z, uu.w), part[h]);
        }
      }
#pragma unroll
      for (int h = 0; h < H; ++h) s_spart[(cq * ROWS + row) * H + h] = part[h].x + part[h].y;
    }
    // ---- (d) E2: h1v = relu(T1 + b1v) -> A0 ----------------------------------------------------------------
    tc::mbar_wait(bar_g2, par);
    tc::tc_fence_after();
    tc::tmem_ld32(t0 + my_t, v);
    tc::tmem_ld_wait();
#pragma unroll
    for (int c8 = 0; c8 < 32; c8 += 8) {
      float o[8];
      const float4 b0 = *reinterpret_cast<const float4*>(s_bias + D + col0 + c8);
      const float4 b1 = *reinterpret_cast<const float4*>(s_bias + D + col0 + c8 + 4);
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int t = 0; t < 8; t += 2) {
        const float2 pre = tc::add2(tc::ld2(v + c8 + t), tc::ld2(bv + t));
        o[t] = fmaxf(pre.x, 0.f); o[t + 1] = fmaxf(pre.y, 0.f);
      }
      tc::st_row8_bf16(sA0, C::ABLK, row, col0 + c8, o);
    }
    tc::tc_fence_before();
    tc::fence_proxy_async();
    __syncthreads();
    if (tid == 0) {
      tc::tc_fence_after();
      issue_gemm<D>(t0, aA0, aW + 2 * C::WIMG, C::ABLK, C::WBLK);
      tc::mma_commit(bar_g3);
    }
    // softmax statistics for this latent (every thread of the row, redundantly; overlaps GEMM3)
    float pw[H], corr[H];
#pragma unroll
    for (int h = 0; h < H; ++h) {
      float dot = 0.f;
#pragma unroll
      for (int q = 0; q < C::NQ; ++q) dot += s_spart[(q * ROWS + row) * H + h];
      float sv = scale * (dot + s_kap[h]) + win;
      if (cq == 0 && row_valid && P.slog) P.slog[((bz * P.C) + c0 + row) * HT + h0 + h] = sv;
      float m_new = fmaxf(m_run[h], sv);
      corr[h] = __expf(m_run[h] - m_new);
      pw[h] = __expf(sv - m_new);
      l_run[h] = l_run[h] * corr[h] + pw[h];
      m_run[h] = m_new;
    }
    uint32_t dgh[16];                          // my 32 columns of the backward's stash gelu'(tpre) (fp16), parked E3 -> E4_0
    // ---- (e) E3: g = gelu(T0 + b'), row statistics, LayerNorm -> A1 ----
    tc::mbar_wait(bar_g3, par);
    tc::tc_fence_after();
    if (H > 1 && !C::kStageAll && tid == 0) {          // A0 is free again: stream W3[z,1] into it
      tc::mbar_expect_tx(&bar_w3[1], C::WIMG);
      tc::bulk_g2s(sA0, P.img_W3 + (bz * HT + h0 + 1) * C::WIMG, C::WIMG, &bar_w3[1]);
    }
    tc::tmem_ld32(t0 + my_t, v);
    tc::tmem_ld_wait();
    {
      float st[2];
      if (P.dgr) gelu_rowsums32_stash(v, s_bias + 2 * D + col0, dgh, st);      // + gelu' of this layer, packed, for the backward
      else gelu_rowsums32(v, s_bias + 2 * D + col0, st);
      xw = 0;
      row_exchange<C::NQ, 2>(s_exch, xw, cq, row, lq, st);
      const float mu = st[0] * (1.f / D);
      const float rstd = rsqrtf(fmaxf(st[1] * (1.f / D) - mu * mu, 0.f) + 1e-6f);
      const float2 rstd2 = tc::splat2(rstd), nm2 = tc::splat2(-mu * rstd);
#pragma unroll
      for (int c8 = 0; c8 < 32; c8 += 8) {
        float o[8];
#pragma unroll
        for (int t = 0; t < 8; t += 2) tc::st2(o + t, tc::fma2(tc::ld2(v + c8 + t), rstd2, nm2));
        tc::st_row8_bf16(sA1, C::ABLK, row, col0 + c8, o);
      }
      if (P.dgr && cq == 0) P.trstd[(size_t)bz * gridDim.x * ROWS + c0 + row] = rstd;
    }
    tc::cp_async_wait_all();                  // the next latent's vectors (requested at the top) are visible after this barrier
    tc::tc_fence_before();
    tc::fence_proxy_async();
    __syncthreads();
    if (tid == 0) {
      if (P.that_img) {                // stash the that operand tile for backward kernel A (bulk store, no thread work)
        tc::bulk_s2g(P.that_img + ((size_t)bz * gridDim.x + blockIdx.x) * C::ATILE, sA1, C::ATILE);
        tc::bulk_commit();
      }
      tc::mbar_wait(&bar_w3[0], par);
      tc::tc_fence_after();
      issue_gemm<D>(t0, aA1, aS, C::ABLK, C::WBLK);
      tc::mma_commit(&bar_g4[0]);
      if (H > 1) {
        if (!C::kStageAll) tc::mbar_wait(&bar_w3[1], par);
        issue_gemm<D>(t1, aA1, C::kStageAll ? aS + C::WIMG : aA0, C::ABLK, C::WBLK);
        tc::mma_commit(&bar_g4[1]);
      }
    }
    // ---- invariants of the NEXT latent -> projection operand, in the shadow of GEMM4_0; warp 0 collects the arrivals and
    //      issues the tiny phase MMA behind GEMM4 (named barrier 6: arrive / sync, nobody else blocks)
    if (more) {
      write_invariants(s_lam_next, par ^ 1);
      tc::fence_proxy_async();
    }
    // ---- (f) E4: per head  m = T + b3 ; n = LN(gelu(m)) ; acc += p n --------------------------------------------
#pragma unroll
    for (int h = 0; h < H; ++h) {
      tc::mbar_wait(&bar_g4[h], par);
      tc::tc_fence_after();
      tc::tmem_ld32(((h & 1) ? t1 : t0) + my_t, v);
      tc::tmem_ld_wait();
      if (h == 0 && (more || P.dgr || H == 3)) {
        // GEMM4_0 is complete, so the W3 stage buffer is free: it stages the backward's stash rstd * gelu' (in kernel B's load
        // order [column quarter][chunk][row] x 16 bytes), which then leaves by ONE bulk store -- 64 STG.128 per CTA in a burst
        // stalled every warp on the SM's store path instead.  T0 has been read by this thread: when everybody has, the next
        // latent's phases land there.
        if (P.dgr) {
          uint4* stage = reinterpret_cast<uint4*>(sG) + cq * 4 * ROWS + row;
#pragma unroll
          for (int q = 0; q < 4; ++q) stage[q * ROWS] = make_uint4(dgh[4 * q], dgh[4 * q + 1], dgh[4 * q + 2], dgh[4 * q + 3]);
          tc::fence_proxy_async();
        }
        tc::tc_fence_before();
        if (warp == 0) {
          tc::named_sync(6, C::NT);
          if (tid == 0) {
            if (more) {
              tc::tc_fence_after();
              issue_proj(tp, aU, aOm, D);
              tc::mma_commit(bar_p);
            }
            if (H == 3) {      // T0 has been read by everybody: the third head's GEMM4 goes there
              issue_gemm<D>(t0, aA1, aS + 2 * C::WIMG, C::ABLK, C::WBLK);
              tc::mma_commit(&bar_g4[2]);
            }
            if (P.dgr) {
              tc::bulk_s2g(P.dgr + ((size_t)bz * gridDim.x + blockIdx.x) * (C::DTILE / 16), sG, C::DTILE);
              tc::bulk_commit();
            }
          }
          __syncwarp();
        } else {
          tc::named_arrive(6, C::NT);
        }
      }
      float st[2];
      gelu_rowsums32(v, s_b3 + h * D + col0, st);
      float a[32];                            // the accumulator slab: requested now, first touched after the exchange
      tc::tmem_ld32(tacc + h * D + my_t, a);
      xw = (h + 1) & 1;                       // E4_0 -> buffer 1 (the logit partials are dead), E4_1 -> buffer 0
      row_exchange<C::NQ, 2>(s_exch, xw, cq, row, lq, st);
      float mu = st[0] * (1.f / D);
      float rstd = rsqrtf(fmaxf(st[1] * (1.f / D) - mu * mu, 0.f) + 1e-6f);
      const float pr = pw[h] * rstd;
      const float2 pr2 = tc::splat2(pr), tz2 = tc::splat2(-pr * mu), corr2 = tc::splat2(corr[h]);
      tc::tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; j += 2) tc::st2(a + j, tc::fma2(tc::ld2(v + j), pr2, tc::fma2(tc::ld2(a + j), corr2, tz2)));
      tc::tmem_st32(tacc + h * D + my_t, a);
    }
    if (tid == 0) {
      if (P.that_img) tc::bulk_wait_read0();   // the stashes have been read out of A1 / the stage buffer before they are overwritten
      if (more) {                              // stage buffer: next latent's W3[.,0] (needed by its GEMM4_0, most of a latent away)
        tc::mbar_expect_tx(&bar_w3[0], C::SBYTES);
        tc::bulk_g2s(sS, P.img_W3 + ((bz + 1) * HT + h0) * C::WIMG, C::SBYTES, &bar_w3[0]);
      }
    }
    tc::tmem_st_wait();
    tc::tc_fence_before();
    __syncthreads();
  }

#pragma unroll
  for (int h = 0; h < H; ++h) {
    float a[32];
    tc::tmem_ld32(tacc + h * D + my_t, a);    // (warp-collective: outside the row_valid branch)
    tc::tmem_ld_wait();
    if (row_valid) {
      float inv_l = 1.f / l_run[h];
      float* o = P.nbar + (((int64_t)b * P.C + c0 + row) * HT + h0 + h) * D + col0;
#pragma unroll
      for (int j = 0; j < 32; j += 4)
        *reinterpret_cast<float4*>(o + j) = make_float4(a[j] * inv_l, a[j + 1] * inv_l, a[j + 2] * inv_l, a[j + 3] * inv_l);
      if (cq == 0) P.lse[((int64_t)b * P.C + c0 + row) * HT + h0 + h] = m_run[h] + logf(l_run[h]);
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc<C::TMEM_COLS>(tm);
}

template <int D, int H, bool G = false>
int launch_tc(cudaStream_t st, const EnfPairTcParams& p, int h0 = 0, int HT = H) {
  using C = TcCfg<D, H>;
  if (cudaFuncSetAttribute(pairs_fwd_tc_kernel<D, H, G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM_BYTES) != cudaSuccess)
    return -1;
  dim3 grid((p.C + ROWS - 1) / ROWS, p.B);
  pairs_fwd_tc_kernel<D, H, G><<<grid, C::NT, C::SMEM_BYTES, st>>>(p, h0, HT);
  return 1;
}

// More heads than one kernel holds in TMEM: one launch per group of at most two heads (H = 3: 2 + 1, H = 4: 2 + 2).  Every
// launch recomputes the shared value and query path; only the first writes the backward's stash, which does not depend on
// the heads.
template <int D>
int launch_tc_groups(cudaStream_t st, int H, const EnfPairTcParams& p) {
  EnfPairTcParams q = p;
  int n = 0;
  for (int h0 = 0; h0 < H; h0 += 2) {
    const int r = H - h0 >= 2 ? launch_tc<D, 2, true>(st, q, h0, H) : launch_tc<D, 1, true>(st, q, h0, H);
    if (r < 0) return -1;
    n += r;
    q.that_img = nullptr; q.dgr = nullptr; q.trstd = nullptr;
  }
  return n;
}

}  // namespace

bool enf_pairs_fwd_tc_supported(int d, int H) { return (d == 128 || d == 64 || d == 32) && H >= 1 && H <= 4; }

int enf_launch_pairs_fwd_tc(cudaStream_t st, int d, int H, const EnfPairTcParams& p) {
  if (d == 32 && H == 4) return launch_tc_groups<32>(st, H, p);
  if (d == 128 && H > 2) return launch_tc_groups<128>(st, H, p);
  if (d == 64 && H > 2) return launch_tc_groups<64>(st, H, p);
  if (d == 32 && H == 3) return launch_tc<32, 3>(st, p);
  if (d == 32 && H == 2) return launch_tc<32, 2>(st, p);
  if (d == 32 && H == 1) return launch_tc<32, 1>(st, p);
  if (d == 128 && H == 2) return launch_tc<128, 2>(st, p);
  if (d == 128 && H == 1) return launch_tc<128, 1>(st, p);
  if (d == 64 && H == 2) return launch_tc<64, 2>(st, p);
  if (d == 64 && H == 1) return launch_tc<64, 1>(st, p);
  return -1;
}
