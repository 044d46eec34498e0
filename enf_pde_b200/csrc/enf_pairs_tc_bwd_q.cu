// Fused (query, latent)-pair BACKWARD, kernel C: the QUERY path and the invariant / window backward
// (EnfPrecision::ENF_PREC_BF16, d = 128).  Runs after kernels A and B of enf_pairs_tc_bwd.cu.
//
// Persistent CTAs walk (field, latent) items; per item they walk the field's query tiles (128 rows each):
//     S1  gamma_q (hi | lo fp16 split) from the RFF phases the tensor core left in TMEM
//     M1  T   = gamma_q W1_q                  (3-term split product, as the relu mask decides whole gradient entries)
//     E   h1q = relu(T + b1q) ; dzq = scale sum_h ds_h U_h [h1q > 0]          -> two fp16 operand tiles
//     M2  S2 += h1q^T [1 | ds]   (dU)     T = dzq W1_q^T (d gamma_q)     dW1_q += gamma_q^T dzq     S1 += dzq^T [1 | ds] (db1q)
//         + RFF phases of the next tile
//     S3  dproj_j = cos_j dsin_j - sin_j dcos_j  (thread-local: a thread owns sin AND cos of its 16 frequencies) -> tile
//     M3  du = dproj Omega^T                  (N = 16: [Omega_hi | Omega_lo])
//     S4  (one thread per row, overlapped with the next tile's M1) du += du_v (kernel B) ; window backward ;
//         dq ; dLam += dq^T xi through a transposing butterfly ; dsigma ; with GX also the cotangent of the row's query
//         record, d xi += dq Lam (reduced over latents in global memory: one vector reduction per row thread and tile)
// Every reduction over query rows that is a matrix product runs on the tensor core: column sums (bias gradient) and
// ds-weighted column sums (dU) are `tile^T x S` MMAs against a [128 rows x 16] side operand S = [1 | ds_hi | ds_lo].
// Shared-weight accumulators (dW1_q, db1q) live in TMEM for the CTA's whole life and are flushed once.
#include "enf_pairs_tc_common.cuh"

namespace {

using namespace tcp;

template <int D, int H> struct QCfg {
  static constexpr int NQ = D / 32;
  static constexpr int NT = ROWS * NQ;
  static constexpr int HD = D / 2;
  static constexpr uint32_t WIMG = wimg_bytes<D>();
  static constexpr uint32_t WBLK = D * 128;
  static constexpr uint32_t ABLK = ROWS * 128;
  static constexpr uint32_t ATILE = atile_bytes<D>();
  // d = 32 has ONE thread per query row, which would leave it all of the per-row side work (next tile's invariants AND both
  // halves of the previous tile's window / invariant backward): four SIDE warps (column quarter NQ) take the row backward
  static constexpr int NSIDE = D == 32 ? ROWS : 0;
  static constexpr int NTALL = NT + NSIDE;
  static constexpr int TMEM_NEED = 2 * D + 64 + 48;           // T | dW1_q | phases (64) | db1q | dU | du (16 each)
  static constexpr int TMEM_COLS = TMEM_NEED <= 256 ? 256 : 512;
  // side operand row [1 | ds_hi (H) | ds_lo (H)]: one 16-byte chunk (8 halves) up to H = 3, both chunks the N = 16 MMAs read at H = 4
  static constexpr int NSIDE_HALVES = 1 + 2 * H <= 8 ? 8 : 16;
  static_assert(1 + 2 * H <= 16, "side operand row: [1 | ds_hi (H) | ds_lo (H)] in 16 halves");
  static constexpr uint32_t OFF_W = 0;                         // W1_q image, W1_q low image
  static constexpr uint32_t OFF_GHI = 2 * WIMG;                // gamma_q hi
  static constexpr uint32_t OFF_GLO = OFF_GHI + ATILE;         // gamma_q lo -> h1q -> dproj
  static constexpr uint32_t OFF_DZ = OFF_GLO + ATILE;          // dzq
  static constexpr uint32_t OFF_S = OFF_DZ + ATILE;            // side operand [128 rows][128 B]
  static constexpr uint32_t OFF_U = OFF_S + ABLK;              // projection operand (invariants), 2 atoms
  static constexpr uint32_t OFF_OM = OFF_U + 2 * kProjAtom;    // Omega_q projection image, 1 atom
  static constexpr uint32_t OFF_OMT = OFF_OM + kProjAtom;      // Omega_q^T image for du, [16][64]
  static constexpr uint32_t OFF_F = OFF_OMT + 2048;
  static constexpr int RX = 20;                                // per-row record: xi[8] | u[6], w, c | dw | pad
  static constexpr int F_TOTAL = 64 /*lam*/ + D /*b1q*/ + H * D /*scale U*/ + 64 /*dlam*/ + 8 /*dkappa*/ + 3 * ROWS * RX /*row records of 3 tiles*/;
  static constexpr uint32_t SMEM_BYTES = OFF_F + F_TOTAL * 4 + 128 + 1024;
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
};

__device__ __forceinline__ void load_scale_q(const float* gmax, float& gs, float& inv_gs) {
  float m = *gmax;
  int e = 0;
  const bool ok = m > 0.f && isfinite(m);
  if (ok) frexpf(m, &e);
  gs = ok ? ldexpf(1.f, 4 - e) : 1.f;
  inv_gs = 1.f / gs;
}

// D[D x 16] (+)= Act^T S : Act = [128 rows][D] activation tile read MN-major (M = feature), S = [128 rows][16] side operand
template <int D>
__device__ __forceinline__ void issue_rowsum(uint32_t d_tmem, uint32_t act_addr, uint32_t s_addr, uint32_t ablk, uint32_t accumulate) {
  constexpr uint32_t idesc = tc::make_idesc(wgrad_m<D>(), 16, tc::kOperandFmt, 1, 1);
#pragma unroll
  for (int kk = 0; kk < ROWS / 16; ++kk)
    tc::mma_f16(d_tmem, tc::desc_mnmajor(act_addr + kk * 2048, ablk), tc::desc_mnmajor(s_addr + kk * 2048, ROWS * 128), idesc,
                (kk > 0) | accumulate);
}
// D[128 x 16] = Dp[128 rows][HD <= 64] (K-major, first feature block) * OmT[16][HD] (K-major)
template <int HD>
__device__ __forceinline__ void issue_du(uint32_t d_tmem, uint32_t a_addr, uint32_t b_addr) {
  constexpr uint32_t idesc = tc::make_idesc(ROWS, 16, tc::kOperandFmt, 0, 0);
#pragma unroll
  for (int kk = 0; kk < HD / 16; ++kk) tc::mma_f16(d_tmem, tc::desc_kmajor(a_addr + kk * 32), tc::desc_kmajor(b_addr + kk * 32), idesc, kk > 0);
}

// *addr += (a, b, c, d) as one 16-byte reduction (addr 16-byte aligned)
__device__ __forceinline__ void red_add_f32x4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// GX: also reduce the cotangent of the query records into P.g_xi (ENF_FLAG_GRAD_X); false compiles to the plain backward
template <int D, int H, bool GX>
__global__ void __launch_bounds__(QCfg<D, H>::NTALL, D <= 64 ? 2 : 1) pairs_bwd_tc_q_kernel(EnfPairTcBwdParams P) {
  using C = QCfg<D, H>;
  constexpr int HD = C::HD;
  constexpr int MMA_TID = C::NT - 128;                // lane 0 of the first warp of the last column quarter
  // per-row side work by column quarter: 0 = next tile's invariants, kPart0 / kPart1 = the two halves of the previous
  // tile's window / invariant backward (at d = 64 a row has two threads: quarter 0 also takes the second half; at d = 32 it
  // has one, which takes everything)
  constexpr bool kSide = C::NSIDE > 0;                // side warps: column quarter NQ does BOTH halves of the row backward
  constexpr int kPart0 = (C::NQ > 1 || kSide) ? 1 : 0, kPart1 = C::NQ > 2 ? 2 : (kSide ? 1 : 0);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sW = base + C::OFF_W;
  uint8_t* sGhi = base + C::OFF_GHI;
  uint8_t* sGlo = base + C::OFF_GLO;
  uint8_t* sDz = base + C::OFF_DZ;
  uint8_t* sS = base + C::OFF_S;
  uint8_t* sU = base + C::OFF_U;
  uint8_t* sOm = base + C::OFF_OM;
  uint8_t* sOmT = base + C::OFF_OMT;
  float* f = reinterpret_cast<float*>(base + C::OFF_F);
  float* s_lam = f; f += 64;
  float* s_b1q = f; f += D;
  float* s_us = f; f += H * D;                        // scale * U[b,z,h,:]
  float* s_dlam = f; f += 64;                         // [0,56): dLam, [56]: dsigma
  float* s_dkap = f; f += 8;
  float* s_rx = f; f += 3 * ROWS * C::RX;             // [3 tiles][ROWS][RX]: query features, invariants, window and dw of a row, written
                                                      // by the row's cq == 0 thread, read one tile later by its cq == 1, 2 threads
  uint64_t* bars = reinterpret_cast<uint64_t*>(f);
  uint64_t *bar_w = bars, *bar_p = bars + 1, *bar_g1 = bars + 2, *bar_d = bars + 3, *bar_u = bars + 4;
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bars + 5);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int lq = warp & 3, cq = warp >> 2;
  const int row = lq * 32 + lane, col0 = cq * 32;
  const bool main_thr = cq < C::NQ;                   // owns 32 accumulator columns (false: a side warp, d = 32 only)
  const float scale = rsqrtf((float)D);
  // row (feature) of an M = D accumulator held by my TMEM lane: M = 128 keeps row r in lane r, M = 64 (d = 64) in lane
  // 32 (r / 16) + r % 16 (tests/test_gpu_tc_primitives.py)
  const int wrow = wgrad_row<D>(row, lq, lane);

  if (tid == 0) {
    for (int i = 0; i < 5; ++i) tc::mbar_init(bars + i, 1);
    tc::mbar_fence_init();
  }
  if (warp == 0) tc::tmem_alloc<C::TMEM_COLS>(s_tmem);
  for (int e = tid; e < D; e += C::NTALL) s_b1q[e] = P.q_b1[e];
  {
    uint4* z4 = reinterpret_cast<uint4*>(sS);          // S, U, Om, OmT are contiguous
    for (int e = tid; e < (int)(C::OFF_F - C::OFF_S) / 16; e += C::NTALL) z4[e] = make_uint4(0u, 0u, 0u, 0u);
  }
  float gs, inv_gs;
  load_scale_q(P.gmax, gs, inv_gs);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tm = *s_tmem;
  const uint32_t tT = tm, tW = tm + D, tP = tm + 2 * D, tS1 = tP + 64, tS2 = tS1 + 16, tDu = tS2 + 16;
  const uint32_t lane_off = (uint32_t)(lq * 32) << 16;
  const uint32_t my_t = lane_off + col0;
  if (tid == MMA_TID) {
    tc::mbar_expect_tx(bar_w, 2 * C::WIMG);
    tc::bulk_g2s(sW, P.img_q_w1, C::WIMG, bar_w);
    tc::bulk_g2s(sW + C::WIMG, P.img_q_w1_lo, C::WIMG, bar_w);
  }
  const uint32_t aW = tc::smem_u32(sW), aWlo = aW + C::WIMG, aGhi = tc::smem_u32(sGhi), aGlo = tc::smem_u32(sGlo),
                 aDz = tc::smem_u32(sDz), aS = tc::smem_u32(sS), aU = tc::smem_u32(sU), aOm = tc::smem_u32(sOm),
                 aOmT = tc::smem_u32(sOmT);
  // Omega images: projection operand (phases) and its transpose for du, both as a two-term fp16 split of 2 pi Omega
  proj_build_omega(sOm, 0, P.q_omega, P.rec.I, HD, tid, C::NTALL);
  for (int e = tid; e < P.rec.I * HD; e += C::NTALL) {
    const int i = e / HD, j = e % HD;
    const float val = 6.283185307179586f * P.q_omega[e];
    const __half hi = __float2half_rn(val);
    const __half lo = __float2half_rn(val - __half2float(hi));
    auto off = [&](int n) { return (uint32_t)((n >> 3) * 1024 + (n & 7) * 128 + ((((j >> 3) ^ (n & 7))) << 4) + (j & 7) * 2); };
    *reinterpret_cast<__half*>(sOmT + off(i)) = hi;
    *reinterpret_cast<__half*>(sOmT + off(6 + i)) = lo;
  }

  const int ntiles = (P.C + ROWS - 1) / ROWS;
  const int nitems = P.B * P.Z;
  uint32_t it = 0;                                     // tiles processed by this CTA (barrier parities)

  for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
    const int64_t bz = item;
    const int b = item / P.Z;
    __syncthreads();                                   // the previous item's flush is done with s_*
    if (tid < ENF_LAM_SIZE) s_lam[tid] = P.lam[bz * ENF_LAM_SIZE + tid];
    if (tid < 64) s_dlam[tid] = 0.f;
    if (tid < 8) s_dkap[tid] = 0.f;
    for (int e = tid; e < H * D; e += C::NTALL) s_us[e] = scale * P.U[bz * H * D + e];
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
    const uint32_t it0 = it;                           // row-record slot of tile ct of this item: (it0 + ct) % 3
    auto write_invariants = [&](int ct, const float* xi_r) {
      const EnfPairRecord rec = pair_record<true>(P.rec, s_lam, xi_r, sigma);
      proj_write_u(sU, row, rec.u, P.rec.I);
      float4* rx = reinterpret_cast<float4*>(s_rx + (((it0 + ct) % 3) * ROWS + row) * C::RX);
      rx[0] = make_float4(xi_r[0], xi_r[1], xi_r[2], xi_r[3]);
      rx[1] = make_float4(xi_r[4], xi_r[5], xi_r[6], xi_r[7]);
      rx[2] = make_float4(rec.u[0], rec.u[1], rec.u[2], rec.u[3]);
      rx[3] = make_float4(rec.u[4], rec.u[5], rec.w, rec.c);
    };
    float lam_acc0 = 0.f, lam_acc1 = 0.f, kap_acc[H];         // lam_acc<part> of the thread that owns `part`: 0: dLam[0..31], 1: dLam[32..55] | dsigma
#pragma unroll
    for (int h = 0; h < H; ++h) kap_acc[h] = 0.f;
    // du (tile ct) + du_v -> window backward -> dq -> my half of dLam / dsigma partial sums (lane l keeps column l).
    // The row's record comes from shared memory (written a tile earlier by the cq == 0 thread); part = 0: cq == 1, 1: cq == 2.
    auto load_duv = [&](int ct, float* duv) {
#pragma unroll
      for (int k = 0; k < 8; ++k) duv[k] = 0.f;
      if (ct * ROWS + row < P.C) {
        const float4* src = reinterpret_cast<const float4*>(P.duv + (bz * P.C + ct * ROWS + row) * 8);
        float4 a = __ldg(src), c = __ldg(src + 1);
        duv[0] = a.x; duv[1] = a.y; duv[2] = a.z; duv[3] = a.w; duv[4] = c.x; duv[5] = c.y; duv[6] = c.z; duv[7] = c.w;
      }
    };
    auto row_backward = [&](int ct, uint32_t par_u, int part, const float* duv) {
      const float4* rx = reinterpret_cast<const float4*>(s_rx + (((it0 + ct) % 3) * ROWS + row) * C::RX);
      const float4 x0 = rx[0], x1 = rx[1], r0 = rx[2], r1 = rx[3];
      const float xi_r[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
      EnfPairRecord rec;
      rec.u[0] = r0.x; rec.u[1] = r0.y; rec.u[2] = r0.z; rec.u[3] = r0.w; rec.u[4] = r1.x; rec.u[5] = r1.y; rec.w = r1.z; rec.c = r1.w;
      const float dw = reinterpret_cast<const float*>(rx)[16];
      tc::mbar_wait(bar_u, par_u);
      tc::tc_fence_after();
      float d16[16];
      tc::tmem_ld16(tDu + lane_off, d16);
      tc::tmem_ld_wait();
      float du[6];
#pragma unroll
      for (int i = 0; i < 6; ++i) du[i] = i < P.rec.I ? d16[i] + d16[6 + i] + duv[i] : 0.f;
      float dq[ENF_R_LAM], dsg;
      record_adjoint(P.rec, rec, du, dw, sigma, dq, dsg);
      if constexpr (GX) {
        // d xi[f] for my half of the record (part 0: f = 0..3, part 1: f = 4..7)
        if (ct * ROWS + row < P.C) {
          float g[4] = {0.f, 0.f, 0.f, 0.f};
          record_xi_cotangent(P.rec, s_lam, xi_r, dq, part, g);
          red_add_f32x4(P.g_xi + ((int64_t)b * P.C + ct * ROWS + row) * ENF_F_XI + 4 * part,
                        g[0] * inv_gs, g[1] * inv_gs, g[2] * inv_gs, g[3] * inv_gs);
        }
      }
      float vv[32];
      if (part == 0) {
#pragma unroll
        for (int e = 0; e < 32; ++e) vv[e] = dq[e >> 3] * xi_r[e & 7];
      } else {
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          const int e1 = 32 + e;
          vv[e] = e1 < ENF_LAM_SIZE ? dq[e1 >> 3] * xi_r[e1 & 7] : (e1 == ENF_LAM_SIZE ? dsg : 0.f);
        }
      }
      const float cs = warp_colsum32(vv, lane);
      if (part == 0) lam_acc0 += cs; else lam_acc1 += cs;
    };

    if (cq == 0) {
      float xi0[8];
      load_xi(0, xi0);
      write_invariants(0, xi0);
    }
    float dsv_next[H];                                  // logit cotangents of the tile about to start (fetched a tile ahead)
#pragma unroll
    for (int h = 0; h < H; ++h) dsv_next[h] = (main_thr && row < P.C) ? __ldg(P.ds + (bz * P.C + row) * H + h) : 0.f;
    tc::fence_proxy_async();
    __syncthreads();
    if (warp == (MMA_TID >> 5)) {
      if (tc::elect_one()) {
        tc::tc_fence_after();
        issue_proj(tP, aU, aOm, HD);
        tc::mma_commit(bar_p);
      }
      __syncwarp();
    }

    for (int ct = 0; ct < ntiles; ++ct, ++it) {
      const uint32_t par = it & 1;
      const int c0 = ct * ROWS;
      const bool valid = c0 + row < P.C;
      const int64_t pr = bz * P.C + c0 + row;
      float dsv[H];
#pragma unroll
      for (int h = 0; h < H; ++h) dsv[h] = dsv_next[h];
      // global operands of this tile's side work, requested before the RFF pass: one row record per thread role
      float pre8[8];                                       // cq == 0: xi of tile ct + 1 ; cq == 1, 2: du_v of tile ct - 1
      if (cq == 0) { if (ct + 1 < ntiles) load_xi(ct + 1, pre8); }
      else if (cq == kPart0 || cq == kPart1) { if (ct > 0) load_duv(ct - 1, pre8); }
      if (it > 0) tc::mbar_wait(bar_u, (it - 1) & 1);     // every MMA of the previous tile is done with the operand tiles
      // ---- S1: gamma_q hi / lo ---------------------------------------------------------------------------------
      tc::mbar_wait(bar_p, par);
      tc::tc_fence_after();
      if (main_thr) rff_from_proj<D, true>(tP + lane_off + 16 * cq, sGhi, sGlo, C::ABLK, row, 16 * cq);
      tc::tc_fence_before();
      tc::fence_proxy_async();
      __syncthreads();
      if (warp == (MMA_TID >> 5)) {
        if (tc::elect_one()) {
          if (it == 0) tc::mbar_wait(bar_w, 0);
          tc::tc_fence_after();
          issue_gemm<D>(tT, aGhi, aW, C::ABLK, C::WBLK);
          issue_gemm<D>(tT, aGlo, aW, C::ABLK, C::WBLK, 1);
          issue_gemm<D>(tT, aGhi, aWlo, C::ABLK, C::WBLK, 1);
          tc::mma_commit(bar_g1);
        }
        __syncwarp();
      }
      // ---- per-row side work, overlapped with the 3-term GEMM: shared by three of the row's four threads ----------------
      if (cq == 0) {
        {                                                  // side operand row: [1 | ds_hi | ds_lo | 0 ...]
          __half hv[C::NSIDE_HALVES];
          hv[0] = __float2half_rn(1.f);
#pragma unroll
          for (int k = 1; k < C::NSIDE_HALVES; ++k) hv[k] = __float2half_rn(0.f);
#pragma unroll
          for (int h = 0; h < H; ++h) {
            hv[1 + h] = __float2half_rn(dsv[h]);
            hv[1 + H + h] = __float2half_rn(dsv[h] - __half2float(hv[1 + h]));
          }
#pragma unroll
          for (int k = 0; k < C::NSIDE_HALVES / 8; ++k)
            *reinterpret_cast<uint4*>(sS + tc::swz_chunk_off(row, k)) = *reinterpret_cast<const uint4*>(hv + 8 * k);
        }
        float dw = 0.f;
#pragma unroll
        for (int h = 0; h < H; ++h) { kap_acc[h] += dsv[h]; dw += dsv[h]; }
        s_rx[(((it0 + ct) % 3) * ROWS + row) * C::RX + 16] = dw;
        if (ct + 1 < ntiles) write_invariants(ct + 1, pre8);
        if (kPart1 == 0 && !kSide && ct > 0) {             // d = 64: this thread also owns the second half of the row backward
          float duv[8];                                    //          (d = 32: both halves)
          load_duv(ct - 1, duv);
          if (kPart0 == 0) row_backward(ct - 1, (it - 1) & 1, 0, duv);
          row_backward(ct - 1, (it - 1) & 1, 1, duv);
        }
      } else if (kSide) {
        if (ct > 0) { row_backward(ct - 1, (it - 1) & 1, 0, pre8); row_backward(ct - 1, (it - 1) & 1, 1, pre8); }
      } else if ((cq == kPart0 || cq == kPart1) && ct > 0) {
        row_backward(ct - 1, (it - 1) & 1, cq == kPart0 ? 0 : 1, pre8);
      }
      // ---- E: h1q, dzq ---------------------------------------------------------------------------------------------
      if (main_thr) {
      float v[32];
      tc::mbar_wait(bar_g1, par);
      tc::tc_fence_after();
      tc::tmem_ld32(tT + my_t, v);
      tc::tmem_ld_wait();
#pragma unroll
      for (int c8 = 0; c8 < 32; c8 += 8) {
        float oh[8], oz[8];
#pragma unroll
        for (int q4 = 0; q4 < 8; q4 += 4) {
          const float4 bb = *reinterpret_cast<const float4*>(s_b1q + col0 + c8 + q4);
          float4 uu[H];
#pragma unroll
          for (int h = 0; h < H; ++h) uu[h] = *reinterpret_cast<const float4*>(s_us + h * D + col0 + c8 + q4);
          const float bv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
          for (int t = 0; t < 4; t += 2) {
            const float2 pre = tc::add2(tc::ld2(v + c8 + q4 + t), tc::ld2(bv + t));
            float2 a = tc::mul2(tc::splat2(dsv[0]), t == 0 ? make_float2(uu[0].x, uu[0].y) : make_float2(uu[0].z, uu[0].w));
#pragma unroll
            for (int h = 1; h < H; ++h) a = tc::fma2(tc::splat2(dsv[h]), t == 0 ? make_float2(uu[h].x, uu[h].y) : make_float2(uu[h].z, uu[h].w), a);
            oh[q4 + t] = fmaxf(pre.x, 0.f); oh[q4 + t + 1] = fmaxf(pre.y, 0.f);
            oz[q4 + t] = pre.x > 0.f ? a.x : 0.f; oz[q4 + t + 1] = pre.y > 0.f ? a.y : 0.f;
          }
        }
        tc::st_row8_bf16(sGlo, C::ABLK, row, col0 + c8, oh);
        tc::st_row8_bf16(sDz, C::ABLK, row, col0 + c8, oz);
      }
      if (ct + 1 < ntiles) {
#pragma unroll
        for (int h = 0; h < H; ++h) dsv_next[h] = (c0 + ROWS + row < P.C) ? __ldg(P.ds + (pr + ROWS) * H + h) : 0.f;
      }
      }   // main_thr
      tc::tc_fence_before();
      tc::fence_proxy_async();
      __syncthreads();
      if (warp == (MMA_TID >> 5)) {
        if (tc::elect_one()) {
          tc::tc_fence_after();
          // dU first: it is the only MMA that reads the h1q tile, which S3 overwrites with dproj as soon as bar_d fires (MMAs
          // complete in issue order, so the dgrad's commit covers it; eight N = 16 MMAs: nothing next to the dgrad)
          issue_rowsum<D>(tS2, aGlo, aS, C::ABLK, ct > 0);           // dU (per item)
          issue_dgrad<D>(tT, aDz, aW, C::ABLK, C::WBLK, 0);          // d gamma_q (S3 waits for it)
          tc::mma_commit(bar_d);
          if (P.g_q_w1) {                                            // latents-only backward (dW = NULL): no shared-weight gradients
            issue_wgrad<D>(tW, aGhi, aDz, C::ABLK, it > 0);          // dW1_q (per CTA)
            issue_rowsum<D>(tS1, aDz, aS, C::ABLK, it > 0);          // db1q (per CTA)
          }
          if (ct + 1 < ntiles) {
            issue_proj(tP, aU, aOm, HD);
            tc::mma_commit(bar_p);
          }
        }
        __syncwarp();
      }
      // ---- S3: d gamma_q -> dproj (my 16 frequencies: sin columns j, cos columns HD + j) ---------------------------
      if (main_thr) {
      tc::mbar_wait(bar_d, par);
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
            const float2 nsn = __half22float2(__hneg2(hs[t])), cs = __half22float2(hc[t]);       // d sin = cos, d cos = -sin
            tc::st2(o + 2 * t, tc::fma2(nsn, tc::ld2(dcs + c8 + 2 * t), tc::mul2(cs, tc::ld2(dsn + c8 + 2 * t))));
          }
          tc::st_row8_bf16(sGlo, C::ABLK, row, col, o);             // h1q's only reader (dU) was issued before the dgrad: it is complete
        }
      }
      }   // main_thr
      tc::tc_fence_before();
      tc::fence_proxy_async();
      __syncthreads();
      if (warp == (MMA_TID >> 5)) {
        if (tc::elect_one()) {
          tc::tc_fence_after();
          issue_du<HD>(tDu, aGlo, aOmT);
          tc::mma_commit(bar_u);
        }
        __syncwarp();
      }
    }
    // ---- item flush --------------------------------------------------------------------------------------------------
    if (cq == kPart0 || cq == kPart1) {
      float duv[8];
      load_duv(ntiles - 1, duv);
#pragma unroll
      for (int part = 0; part < 2; ++part) {
        if (cq != (part == 0 ? kPart0 : kPart1)) continue;
        row_backward(ntiles - 1, (it - 1) & 1, part, duv);
        atomicAdd(&s_dlam[part * 32 + lane], part == 0 ? lam_acc0 : lam_acc1);
      }
    }
    {
      tc::mbar_wait(bar_u, (it - 1) & 1);
      tc::tc_fence_after();
      if (cq == 0) {
#pragma unroll
        for (int h = 0; h < H; ++h) {
          const float sk = warp_sum(kap_acc[h]);
          if (lane == 0) atomicAdd(&s_dkap[h], sk);
        }
      }
    }
    if (cq == 0) {                                         // dU[h][j], j = the accumulator row of my TMEM lane
      float d16[16];
      tc::tmem_ld16(tS2 + lane_off, d16);
      tc::tmem_ld_wait();
      if (wrow >= 0) {
#pragma unroll
        for (int h = 0; h < H; ++h) P.g_U[bz * H * D + h * D + wrow] = scale * inv_gs * (d16[1 + h] + d16[1 + H + h]);
      }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (tid < ENF_LAM_SIZE) P.g_lam[bz * ENF_LAM_SIZE + tid] = s_dlam[tid] * inv_gs;
    if (tid == ENF_LAM_SIZE && P.rec.win_kind != ENF_WIN_NONE) P.g_sigma[bz] = s_dlam[ENF_LAM_SIZE] * inv_gs;
    if (tid < H) P.g_kappa[bz * H + tid] = scale * inv_gs * s_dkap[tid];
  }
  // ---- CTA flush: shared-weight gradients --------------------------------------------------------------------------------
  __syncthreads();
  tc::tc_fence_after();
  if (it > 0 && main_thr && P.g_q_w1) {
    float v[32];
    tc::tmem_ld32(tW + my_t, v);
    tc::tmem_ld_wait();
    if (wrow >= 0) {
      float* o = P.g_q_w1 + (size_t)wrow * D + col0;
#pragma unroll
      for (int j = 0; j < 32; ++j) atomicAdd(o + j, v[j] * inv_gs);
    }
    if (cq == 0) {
      float d16[16];
      tc::tmem_ld16(tS1 + lane_off, d16);
      tc::tmem_ld_wait();
      if (wrow >= 0) atomicAdd(P.g_q_b1 + wrow, d16[0] * inv_gs);
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc<C::TMEM_COLS>(tm);
}

template <int D, int H, bool GX>
int launch_q(cudaStream_t st, const EnfPairTcBwdParams& p) {
  using C = QCfg<D, H>;
  if (cudaFuncSetAttribute(pairs_bwd_tc_q_kernel<D, H, GX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM_BYTES) != cudaSuccess) return -1;
  int nitems = p.B * p.Z;
  // persistent CTAs: as many as are resident at once.  TMEM (not visible to the occupancy API, which also under-reports
  // kernels with > 48 KB of dynamic shared memory: it answered 1 for d = 32 and halved the grid) allows 512 / TMEM_COLS
  const int occ = D == 32 ? 512 / C::TMEM_COLS : 1;
  int nsm = 148;
  { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev); }
  const int ctas = occ * nsm;
  int grid = nitems < ctas ? nitems : ctas;
  pairs_bwd_tc_q_kernel<D, H, GX><<<grid, C::NTALL, C::SMEM_BYTES, st>>>(p);
  return 1;
}
template <int D, int H>
int launch_q(cudaStream_t st, const EnfPairTcBwdParams& p) { return p.g_xi ? launch_q<D, H, true>(st, p) : launch_q<D, H, false>(st, p); }

}  // namespace

int enf_launch_pairs_bwd_tc_q(cudaStream_t st, int d, int H, const EnfPairTcBwdParams& p) {
  if (d == 32 && H == 4) return launch_q<32, 4>(st, p);
  if (d == 128 && H == 4) return launch_q<128, 4>(st, p);
  if (d == 128 && H == 3) return launch_q<128, 3>(st, p);
  if (d == 64 && H == 4) return launch_q<64, 4>(st, p);
  if (d == 64 && H == 3) return launch_q<64, 3>(st, p);
  if (d == 32 && H == 3) return launch_q<32, 3>(st, p);
  if (d == 32 && H == 2) return launch_q<32, 2>(st, p);
  if (d == 32 && H == 1) return launch_q<32, 1>(st, p);
  if (d == 128 && H == 2) return launch_q<128, 2>(st, p);
  if (d == 128 && H == 1) return launch_q<128, 1>(st, p);
  if (d == 64 && H == 2) return launch_q<64, 2>(st, p);
  if (d == 64 && H == 1) return launch_q<64, 1>(st, p);
  return -1;
}
