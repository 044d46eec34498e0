// Device code shared by the tensor-core pair kernels (forward + the two backward kernels), so that the
// backward's recompute reproduces the forward's operand roundings bit for bit.
//
// Thread layout of every kernel here: a CTA owns 128 query rows (= the 128 TMEM lanes).  NQ = D/32 threads
// serve one row, 32 accumulator columns each: warp w -> lane quadrant lq = w & 3 (rows 32*lq .. +31, the only
// TMEM lanes that warp may touch), column quarter cq = w >> 2 (columns 32*cq .. +31).
#pragma once
#include "enf_common.cuh"
#include "enf_tc.cuh"

namespace tcp {

constexpr int ROWS = 128;

// Operand geometry.  An operand row holds the features in 64-element (128-byte, swizzled) blocks.  num_hidden = 32 keeps
// that row pitch and uses the first half of its single block (tests/test_gpu_tc_primitives.py pins that K-major reads with two
// K-steps, MN-major reads with N = 32 and the M = 64 weight-gradient shape all work on such rows); whatever a kernel leaves in
// the unused half only ever reaches accumulator rows / columns that are never read back.
template <int D> __host__ __device__ constexpr int nblk() { return D >= 64 ? D / 64 : 1; }
template <int D> __host__ __device__ constexpr uint32_t wimg_bytes() { return (uint32_t)nblk<D>() * D * 128; }      // weight image [nblk][D rows][128 B]
template <int D> __host__ __device__ constexpr uint32_t atile_bytes() { return (uint32_t)nblk<D>() * ROWS * 128; }  // activation tile [nblk][128 rows][128 B]
template <int D> __host__ __device__ constexpr int wgrad_m() { return D >= 64 ? D : 64; }                            // M of the weight-gradient MMAs
// weight-gradient accumulator row (input feature) held by a thread's TMEM lane: M = 128 keeps row r in lane r, M = 64 in lane
// 32 (r / 16) + r % 16 (tests/test_gpu_tc_primitives.py); -1: this lane holds no valid row
template <int D> __device__ __forceinline__ int wgrad_row(int row, int lq, int lane) {
  if (D == 128) return row;
  const int r = lane < 16 ? 16 * lq + lane : -1;
  return r < D ? r : -1;
}

__device__ __forceinline__ float tanh_fast(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// v[j] <- g_j = gelu(v[j] + bias[j]) over a thread's 32 columns (bias: 16-byte aligned, shared memory); st = {sum g, sum g^2}
// (even / odd partial sums); gelu is jax.nn.gelu(approximate=True).  The LayerNorm statistics of the forward (E3, E4) in packed form, eight columns at a time and
// stage by stage, so that four independent chains (and their eight MUFU.TANH) are in flight per warp.
__device__ __forceinline__ void gelu_rowsums32(float (&v)[32], const float* bias, float (&st)[2]) {
  const float c0 = 0.7978845608028654f, c1 = 0.7978845608028654f * 0.044715f;
  float2 s0 = tc::splat2(0.f), s1 = tc::splat2(0.f);
#pragma unroll
  for (int c8 = 0; c8 < 32; c8 += 8) {
    const float4 b0 = *reinterpret_cast<const float4*>(bias + c8), b1 = *reinterpret_cast<const float4*>(bias + c8 + 4);
    float2 x[4], p[4];
    x[0] = tc::add2(tc::ld2(v + c8), make_float2(b0.x, b0.y)); x[1] = tc::add2(tc::ld2(v + c8 + 2), make_float2(b0.z, b0.w));
    x[2] = tc::add2(tc::ld2(v + c8 + 4), make_float2(b1.x, b1.y)); x[3] = tc::add2(tc::ld2(v + c8 + 6), make_float2(b1.z, b1.w));
#pragma unroll
    for (int i = 0; i < 4; ++i) p[i] = tc::mul2(x[i], x[i]);
#pragma unroll
    for (int i = 0; i < 4; ++i) p[i] = tc::fma2(tc::splat2(c1), p[i], tc::splat2(c0));
#pragma unroll
    for (int i = 0; i < 4; ++i) p[i] = tc::mul2(x[i], p[i]);
#pragma unroll
    for (int i = 0; i < 4; ++i) { p[i].x = tanh_fast(p[i].x); p[i].y = tanh_fast(p[i].y); }
#pragma unroll
    for (int i = 0; i < 4; ++i) p[i] = tc::fma2(tc::splat2(0.5f), p[i], tc::splat2(0.5f));
#pragma unroll
    for (int i = 0; i < 4; ++i) { x[i] = tc::mul2(x[i], p[i]); tc::st2(v + c8 + 2 * i, x[i]); }
#pragma unroll
    for (int i = 0; i < 4; ++i) { s0 = tc::add2(s0, x[i]); s1 = tc::fma2(x[i], x[i], s1); }
  }
  st[0] = s0.x + s0.y; st[1] = s1.x + s1.y;
}

// The forward's E3 when the backward's stash is requested: as gelu_rowsums32, plus dgh[j/2] <- gelu'(v[j] + bias[j]) packed to
// fp16 on the spot (16 registers; the fp32 derivative is never held).  g and the row sums are bit-identical to gelu_rowsums32.
__device__ __forceinline__ void gelu_rowsums32_stash(float (&v)[32], const float* bias, uint32_t (&dgh)[16], float (&st)[2]) {
  const float c0 = 0.7978845608028654f, c1 = 0.7978845608028654f * 0.044715f;
  float2 s0 = tc::splat2(0.f), s1 = tc::splat2(0.f);
#pragma unroll
  for (int c8 = 0; c8 < 32; c8 += 8) {
    const float4 b0 = *reinterpret_cast<const float4*>(bias + c8), b1 = *reinterpret_cast<const float4*>(bias + c8 + 4);
    float2 x[4], x2[4], p[4];
    x[0] = tc::add2(tc::ld2(v + c8), make_float2(b0.x, b0.y)); x[1] = tc::add2(tc::ld2(v + c8 + 2), make_float2(b0.z, b0.w));
    x[2] = tc::add2(tc::ld2(v + c8 + 4), make_float2(b1.x, b1.y)); x[3] = tc::add2(tc::ld2(v + c8 + 6), make_float2(b1.z, b1.w));
#pragma unroll
    for (int i = 0; i < 4; ++i) x2[i] = tc::mul2(x[i], x[i]);
#pragma unroll
    for (int i = 0; i < 4; ++i) p[i] = tc::fma2(tc::splat2(c1), x2[i], tc::splat2(c0));
#pragma unroll
    for (int i = 0; i < 4; ++i) p[i] = tc::mul2(x[i], p[i]);
#pragma unroll
    for (int i = 0; i < 4; ++i) { p[i].x = tanh_fast(p[i].x); p[i].y = tanh_fast(p[i].y); }
#pragma unroll
    for (int i = 0; i < 4; ++i) x2[i] = tc::fma2(tc::splat2(3.f * c1), x2[i], tc::splat2(c0));      // in the shadow of the tanh
#pragma unroll
    for (int i = 0; i < 4; ++i) p[i] = tc::fma2(tc::splat2(0.5f), p[i], tc::splat2(0.5f));          // s
#pragma unroll
    for (int i = 0; i < 4; ++i) { x[i] = tc::mul2(x[i], p[i]); tc::st2(v + c8 + 2 * i, x[i]); }       // g
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 d = tc::fma2(tc::mul2(x[i], tc::fma2(tc::splat2(-2.f), p[i], tc::splat2(2.f))), x2[i], p[i]);
      dgh[(c8 >> 1) + i] = tc::pack_bf16(d.x, d.y);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) { s0 = tc::add2(s0, x[i]); s1 = tc::fma2(x[i], x[i], s1); }
  }
  st[0] = s0.x + s0.y; st[1] = s1.x + s1.y;
}

// cos of two RFF phases on the FMA pipe (packed), so that the XU pipe (4 lanes per scheduler: a warp-wide MUFU takes 8
// cycles) only evaluates the sines: k = rint(ph / pi) by the magic-number add, r = ph - k pi (two-term Cody-Waite),
// cos(ph) = (-1)^k P(r^2) with a degree-4 fit of cos(sqrt(y)) on [0, (pi/2)^2].  |error| <= 2.2e-7 for |ph| <= 300
// (MUFU.COS: 3.6e-7 inside [-pi, pi], growing with |ph|).  Every kernel takes gamma from these helpers, so the
// backward's recompute reproduces the forward's features bit for bit.
__device__ __forceinline__ float2 cos2_fma(float2 ph) {
  const float kMagic = 12582912.f;                      // 1.5 * 2^23: bit 0 of the sum is the parity of k
  const float2 t = tc::fma2(ph, tc::splat2(0.318309886f), tc::splat2(kMagic));
  const float2 k = tc::add2(t, tc::splat2(-kMagic));
  float2 r = tc::fma2(k, tc::splat2(-3.14159274f), ph);
  r = tc::fma2(k, tc::splat2(8.74227766e-8f), r);        // pi = 3.14159274f - 8.74227766e-8
  const float2 y = tc::mul2(r, r);
  float2 p = tc::fma2(y, tc::splat2(2.3121236154111102e-05f), tc::splat2(-0.001385227427817881f));
  p = tc::fma2(y, p, tc::splat2(0.04166339337825775f));
  p = tc::fma2(y, p, tc::splat2(-0.4999989867210388f));
  p = tc::fma2(y, p, tc::splat2(0.9999999403953552f));
  return make_float2(__uint_as_float(__float_as_uint(p.x) ^ (__float_as_uint(t.x) << 31)),
                     __uint_as_float(__float_as_uint(p.y) ^ (__float_as_uint(t.y) << 31)));
}

// gamma(u) = [sin(2 pi u Omega) | cos(2 pi u Omega)] (rff.py:84-93)
// ---- RFF projection on the tensor core ---------------------------------------------------------------------------
// proj[row][n] = 2 pi sum_i u[row][i] Omega[i][n] as ONE small MMA per 128-row tile (M = 128, N = #frequencies, K = 32)
// instead of I FMAs + I shared loads per output element.  fp16 operands carry a two-term split of both factors so the
// phase keeps fp32-level accuracy:   k 0..5: u_hi * Om_hi    k 6..11: u_lo * Om_hi    k 12..17: u_hi * Om_lo   (rest 0).
// Both operands are MN-major, 128-byte-swizzled tiles of [32 k-rows][64 halves] per 64-wide atom:
//   sU  [2 atoms][32][128 B]  (8 KB)   written per tile by one thread per query row,
//   sOm [N/64 atoms][32][128 B]        built once per CTA.
constexpr uint32_t kProjAtom = 32 * 128;
__device__ __forceinline__ uint32_t proj_elem_off(int k, int m) {      // byte offset of element (k-row k, MN index m)
  return (uint32_t)((m >> 6) * kProjAtom + k * 128 + ((((m & 63) >> 3) ^ (k & 7)) << 4) + (m & 7) * 2);
}
__device__ __forceinline__ void proj_store_pair(uint8_t* tile, int i, int m, float val, bool a_side) {
  const __half hi = __float2half_rn(val);
  const __half lo = __float2half_rn(val - __half2float(hi));
  *reinterpret_cast<__half*>(tile + proj_elem_off(i, m)) = hi;
  *reinterpret_cast<__half*>(tile + proj_elem_off(6 + i, m)) = a_side ? lo : hi;
  *reinterpret_cast<__half*>(tile + proj_elem_off(12 + i, m)) = a_side ? hi : lo;
}
// zero a projection operand tile (all threads), before the first write
__device__ __forceinline__ void proj_zero(uint8_t* tile, int natoms, int tid, int nt) {
  uint4* p = reinterpret_cast<uint4*>(tile);
  for (int e = tid; e < natoms * (int)kProjAtom / 16; e += nt) p[e] = make_uint4(0u, 0u, 0u, 0u);
}
// Omega image: column n of the tile = frequency j of embedding `omega` (I x HD, row-major), scaled by 2 pi
__device__ __forceinline__ void proj_build_omega(uint8_t* tile, int n0, const float* __restrict__ omega, int I, int HD, int tid, int nt) {
  for (int e = tid; e < I * HD; e += nt) {
    const int i = e / HD, j = e % HD;
    proj_store_pair(tile, i, n0 + j, 6.283185307179586f * omega[e], false);
  }
}
__device__ __forceinline__ void proj_write_u(uint8_t* tile, int row, const float* u, int I) {
#pragma unroll
  for (int i = 0; i < 6; ++i) if (i < I) proj_store_pair(tile, i, row, u[i], true);
}
// D[128 x N] = sU^T sOm  (N = 64 or 128)
__device__ __forceinline__ void issue_proj(uint32_t d_tmem, uint32_t u_addr, uint32_t om_addr, int N) {
  const uint32_t idesc = tc::make_idesc(ROWS, N, tc::kOperandFmt, 1, 1);
  const uint32_t a = tc::desc_lo_mn(u_addr, kProjAtom), b = tc::desc_lo_mn(om_addr, kProjAtom);
#pragma unroll
  for (int kk = 0; kk < 2; ++kk) tc::mma_f16_lo(d_tmem, a + kk * (2048 >> 4), b + kk * (2048 >> 4), idesc, kk > 0);
}
// my 16 phases (TMEM columns t_proj .. +15 of my lane) -> sin | cos -> 16-bit, swizzled A tile: columns j0.. and HD + j0..
// SPLIT: also the low part of a two-term 16-bit split into tile_lo.
template <int D, bool SPLIT>
__device__ __forceinline__ void rff_from_proj(uint32_t t_proj, uint8_t* tile_hi, uint8_t* tile_lo, uint32_t ablk, int row, int j0) {
  constexpr int HD = D / 2;
  float ph[16];
  tc::tmem_ld16(t_proj, ph);
  tc::tmem_ld_wait();
#pragma unroll
  for (int c8 = 0; c8 < 16; c8 += 8) {
    float sn[8], cs[8];
#pragma unroll
    for (int t = 0; t < 8; t += 2) {
      sn[t] = __sinf(ph[c8 + t]); sn[t + 1] = __sinf(ph[c8 + t + 1]);
#ifdef ENF_COS_MUFU_SPLIT
      if (SPLIT) { cs[t] = __cosf(ph[c8 + t]); cs[t + 1] = __cosf(ph[c8 + t + 1]); } else
#endif
      tc::st2(cs + t, cos2_fma(tc::ld2(ph + c8 + t)));
    }
    tc::st_row8_bf16(tile_hi, ablk, row, j0 + c8, sn);
    tc::st_row8_bf16(tile_hi, ablk, row, HD + j0 + c8, cs);
    if (SPLIT) {
#pragma unroll
      for (int t = 0; t < 8; ++t) { sn[t] -= tc::round_operand(sn[t]); cs[t] -= tc::round_operand(cs[t]); }
      tc::st_row8_bf16(tile_lo, ablk, row, j0 + c8, sn);
      tc::st_row8_bf16(tile_lo, ablk, row, HD + j0 + c8, cs);
    }
  }
}

// SIN = true: only the sin columns (feature block 0 at D = 128), false: only the cos columns -- lets the MMAs over the
// first half of K start while the second half of gamma is still being evaluated
template <int D, bool SPLIT, bool SIN>
__device__ __forceinline__ void rff_half_from_proj(uint32_t t_proj, uint8_t* tile_hi, uint8_t* tile_lo, uint32_t ablk, int row, int j0) {
  constexpr int HD = D / 2;
  float ph[16];
  tc::tmem_ld16(t_proj, ph);
  tc::tmem_ld_wait();
#pragma unroll
  for (int c8 = 0; c8 < 16; c8 += 8) {
    float v[8];
#pragma unroll
    for (int t = 0; t < 8; t += 2) {
      if (SIN) { v[t] = __sinf(ph[c8 + t]); v[t + 1] = __sinf(ph[c8 + t + 1]); }
#ifdef ENF_COS_MUFU_SPLIT
      else if (SPLIT) { v[t] = __cosf(ph[c8 + t]); v[t + 1] = __cosf(ph[c8 + t + 1]); }
#endif
      else tc::st2(v + t, cos2_fma(tc::ld2(ph + c8 + t)));
    }
    tc::st_row8_bf16(tile_hi, ablk, row, (SIN ? 0 : HD) + j0 + c8, v);
    if (SPLIT) {
#pragma unroll
      for (int t = 0; t < 8; ++t) v[t] -= tc::round_operand(v[t]);
      tc::st_row8_bf16(tile_lo, ablk, row, (SIN ? 0 : HD) + j0 + c8, v);
    }
  }
}

// K-steps [kk0, kk1) of issue_gemm (16 features each)
template <int D>
__device__ __forceinline__ void issue_gemm_ksteps(uint32_t d_tmem, uint32_t a_addr, uint32_t b_addr, uint32_t ablk, uint32_t wblk, int kk0,
                                                  int kk1, uint32_t accumulate_first) {
  constexpr uint32_t idesc = tc::make_idesc(ROWS, D, tc::kOperandFmt, 0, 0);
  const uint32_t a = tc::desc_lo_k(a_addr), b = tc::desc_lo_k(b_addr);
#pragma unroll
  for (int kk = 0; kk < D / 16; ++kk)
    if (kk >= kk0 && kk < kk1)
      tc::mma_f16_lo(d_tmem, a + (((kk >> 2) * ablk + (kk & 3) * 32) >> 4), b + (((kk >> 2) * wblk + (kk & 3) * 32) >> 4), idesc,
                     (kk > kk0) | accumulate_first);
}

// D[128 x N=D] = A[128 x K=D] (K-major activation tile) * B (K-major weight image: rows = output feature)
template <int D>
__device__ __forceinline__ void issue_gemm(uint32_t d_tmem, uint32_t a_addr, uint32_t b_addr, uint32_t ablk, uint32_t wblk, uint32_t accumulate = 0) {
  constexpr uint32_t idesc = tc::make_idesc(ROWS, D, tc::kOperandFmt, 0, 0);
  const uint32_t a = tc::desc_lo_k(a_addr), b = tc::desc_lo_k(b_addr);
#pragma unroll
  for (int kk = 0; kk < D / 16; ++kk)
    tc::mma_f16_lo(d_tmem, a + (((kk >> 2) * ablk + (kk & 3) * 32) >> 4), b + (((kk >> 2) * wblk + (kk & 3) * 32) >> 4), idesc,
                   (kk > 0) | accumulate);
}
// dgrad: D[128 x D] (+)= G[128 x D] * W^T, with the SAME weight image read MN-major (rows = reduction index)
template <int D>
__device__ __forceinline__ void issue_dgrad(uint32_t d_tmem, uint32_t g_addr, uint32_t w_addr, uint32_t ablk, uint32_t wblk, uint32_t accumulate) {
  constexpr uint32_t idesc = tc::make_idesc(ROWS, D, tc::kOperandFmt, 0, 1);
  const uint32_t a = tc::desc_lo_k(g_addr), b = tc::desc_lo_mn(w_addr, wblk);
#pragma unroll
  for (int kk = 0; kk < D / 16; ++kk)
    tc::mma_f16_lo(d_tmem, a + (((kk >> 2) * ablk + (kk & 3) * 32) >> 4), b + kk * (2048 >> 4), idesc, (kk > 0) | accumulate);
}
// wgrad: dW[D x D] (+)= Act[128 x D]^T * G[128 x D]; both activation tiles read MN-major (rows = reduction index)
template <int D>
__device__ __forceinline__ void issue_wgrad(uint32_t d_tmem, uint32_t act_addr, uint32_t g_addr, uint32_t ablk, uint32_t accumulate) {
  constexpr uint32_t idesc = tc::make_idesc(wgrad_m<D>(), D, tc::kOperandFmt, 1, 1);
  const uint32_t a = tc::desc_lo_mn(act_addr, ablk), b = tc::desc_lo_mn(g_addr, ablk);
#pragma unroll
  for (int kk = 0; kk < ROWS / 16; ++kk) tc::mma_f16_lo(d_tmem, a + kk * (2048 >> 4), b + kk * (2048 >> 4), idesc, (kk > 0) | accumulate);
}

// Sum NV per-thread partials over the NQ threads that share a query row.  `buf` = two alternating
// [NQ][ROWS][NV] buffers (toggle `which` on every call); the NQ warps of a lane quadrant meet on named barrier 1+lq.
template <int NQ, int NV>
__device__ __forceinline__ void row_exchange(float* buf, int& which, int cq, int row, int lq, float (&v)[NV]) {
  float* b = buf + which * (NQ * ROWS * NV);
  which ^= 1;
#pragma unroll
  for (int i = 0; i < NV; ++i) b[(cq * ROWS + row) * NV + i] = v[i];
  asm volatile("bar.sync %0, %1;" ::"r"(1 + lq), "r"(32 * NQ) : "memory");
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    float s = 0.f;
#pragma unroll
    for (int q = 0; q < NQ; ++q) s += b[(q * ROWS + row) * NV + i];
    v[i] = s;
  }
}

// v[j] = this lane's (row's) value for column j of its 32-column slab.  Returns, in lane l, the sum over the
// warp's 32 rows of column l (a transposing butterfly: 31 shuffles).  Destroys v.
__device__ __forceinline__ float warp_colsum32(float (&v)[32], int lane) {
#pragma unroll
  for (int half = 16; half >= 1; half >>= 1) {
    const bool upper = (lane & half) != 0;
#pragma unroll
    for (int i = 0; i < half; ++i) {
      float send = upper ? v[i] : v[i + half];
      float keep = upper ? v[i + half] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, half);
    }
  }
  return v[0];
}

// Same for 32 columns held as 16 packed fp16 pairs (word i = columns 2i, 2i + 1 of this lane's row; the operand words an
// activation tile is written with): 16 shuffles instead of 31 -- SHFL runs at one warp instruction per two clocks per SM, so the
// fp32 butterfly costs ~1 k cycles per CTA-wide call.  Sums of 32 fp16 values in fp16 (each call's result is then accumulated
// in fp32 by the caller; measured: the gradients move by no more than the variant that finishes the last three levels in fp32).
// Returns column `lane`'s sum.  Destroys w.
__device__ __forceinline__ float warp_colsum32_h2(uint32_t (&w)[16], int lane) {
  static_assert(tc::kOperandFmt == 0, "the packed words are fp16 pairs");
#pragma unroll
  for (int half = 8; half >= 1; half >>= 1) {
    const bool upper = (lane & (2 * half)) != 0;
#pragma unroll
    for (int i = 0; i < half; ++i) {
      const uint32_t send = upper ? w[i] : w[i + half];
      const uint32_t keep = upper ? w[i + half] : w[i];
      const uint32_t got = __shfl_xor_sync(0xffffffffu, send, 2 * half);
      const __half2 sum = __hadd2(*reinterpret_cast<const __half2*>(&keep), *reinterpret_cast<const __half2*>(&got));
      w[i] = *reinterpret_cast<const uint32_t*>(&sum);
    }
  }
  const uint32_t other = __shfl_xor_sync(0xffffffffu, w[0], 1);
  const float2 tot = __half22float2(__hadd2(*reinterpret_cast<const __half2*>(&w[0]), *reinterpret_cast<const __half2*>(&other)));
  return (lane & 1) ? tot.y : tot.x;
}

}  // namespace tcp
