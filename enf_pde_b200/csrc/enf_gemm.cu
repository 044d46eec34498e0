// Generic strided / batched / split-K fp32 GEMM used by the per-latent (L), per-weight (W) and
// per-query tail (Q) stages.  These stages are a few percent of the work of the fused pair kernels;
// this kernel favours generality (arbitrary strides => transposes and head-sliced views for free)
// over peak throughput.  64x64x16 tiles, 256 threads, 4x4 register tile per thread, 8-stage cp.async pipeline
// (most calls are tiny fold / unfold products whose time is global-load latency, not flops).
#include "enf_common.cuh"

namespace {

constexpr int BM = 64, BN = 64, BK = 16;

struct GemmKArgs {
  const float* A; int64_t sam, sak, sab;
  const float* B; int64_t sbk, sbn, sbb;
  float* C; int64_t scm, scn, scb;
  const float* bias; int64_t bias_bs;
  const float* aux;
  float* C2;
  int round_out;
  int M, N, K, splitk, kchunk;
  int act_a, accumulate;
  float alpha;
};

constexpr int ST = 8;      // cp.async pipeline depth (K = 128 is entirely in flight at once): the small fold / unfold products are
                           // latency bound, not flop bound.  8 stages of A and B tiles = 68 KB of dynamic shared memory

__device__ __forceinline__ void cp_async4(float* dst_smem, const float* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ void gemm_tile(const GemmKArgs& g, int bx, int by, int bzz) {
  extern __shared__ __align__(16) float gemm_smem[];
  float (*As)[BK][BM + 4] = reinterpret_cast<float (*)[BK][BM + 4]>(gemm_smem);
  float (*Bs)[BK][BN + 4] = reinterpret_cast<float (*)[BK][BN + 4]>(gemm_smem + ST * BK * (BM + 4));
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int m0 = bx * BM, n0 = by * BN;
  const int bz = bzz / g.splitk, ks = bzz % g.splitk;
  const float* A = g.A + (int64_t)bz * g.sab;
  const float* B = g.B + (int64_t)bz * g.sbb;
  float* C = g.C + (int64_t)bz * g.scb;
  const int kbeg = ks * g.kchunk;
  const int kend = min(g.K, kbeg + g.kchunk);
  const bool a_kfast = (g.sak == 1);     // consecutive threads walk k (row-major A) else walk m
  const bool b_nfast = (g.sbn == 1);

  // element e = tid + 256 i of a BK x BM (BK x BN) tile: the (k, m) / (k, n) slot this thread fills
  int a_kk[4], a_mm[4], b_kk[4], b_nn[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int e = tid + i * 256;
    if (a_kfast) { a_kk[i] = e & (BK - 1); a_mm[i] = e >> 4; } else { a_mm[i] = e & (BM - 1); a_kk[i] = e >> 6; }
    if (b_nfast) { b_nn[i] = e & (BN - 1); b_kk[i] = e >> 6; } else { b_kk[i] = e & (BK - 1); b_nn[i] = e >> 4; }
  }
  auto load_tile = [&](int stage, int k0) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int gm = m0 + a_mm[i], gk = k0 + a_kk[i];
      float* dst = &As[stage][a_kk[i]][a_mm[i]];
      if (gm < g.M && gk < kend) cp_async4(dst, A + (int64_t)gm * g.sam + (int64_t)gk * g.sak); else *dst = 0.f;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int gn = n0 + b_nn[i], gk = k0 + b_kk[i];
      float* dst = &Bs[stage][b_kk[i]][b_nn[i]];
      if (gn < g.N && gk < kend) cp_async4(dst, B + (int64_t)gk * g.sbk + (int64_t)gn * g.sbn); else *dst = 0.f;
    }
  };

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const int nk = (kend - kbeg + BK - 1) / BK;
#pragma unroll
  for (int s = 0; s < ST - 1; ++s) {
    if (s < nk) load_tile(s, kbeg + s * BK);
    cp_async_commit();
  }
  for (int t = 0; t < nk; ++t) {
    const int stage = t % ST;
    cp_async_wait<ST - 2>();                  // this thread's copies of tile t have landed
    if (g.act_a) {                            // gelu on load, applied by the thread that fetched the element
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float* p = &As[stage][a_kk[i]][a_mm[i]];
        *p = enf_gelu(*p);
      }
    }
    __syncthreads();                          // tile t visible to all; everyone is done computing on tile t - 1
    if (t + ST - 1 < nk) load_tile((t + ST - 1) % ST, kbeg + (t + ST - 1) * BK);
    cp_async_commit();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float4 a = *reinterpret_cast<const float4*>(&As[stage][kk][ty * 4]);
      float4 b = *reinterpret_cast<const float4*>(&Bs[stage][kk][tx * 4]);
      float av[4] = {a.x, a.y, a.z, a.w};
      float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
  }

  const float* bias = g.bias ? g.bias + (int64_t)bz * g.bias_bs : nullptr;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int gm = m0 + ty * 4 + i;
    if (gm >= g.M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int gn = n0 + tx * 4 + j;
      if (gn >= g.N) continue;
      float v = g.alpha * acc[i][j];
      if (bias && ks == 0) v += bias[gn];
      int64_t off = (int64_t)gm * g.scm + (int64_t)gn * g.scn;
      if (g.aux) v *= enf_gelu_grad(g.aux[(int64_t)bz * g.scb + off]);
      if (g.accumulate) atomicAdd(C + off, v); else C[off] = enf_maybe_round(v, g.round_out);
      if (g.C2) g.C2[(int64_t)bz * g.scb + off] = enf_maybe_round(enf_gelu(v), g.round_out);
    }
  }
}

__global__ void __launch_bounds__(256) enf_gemm_kernel(const __grid_constant__ GemmKArgs g) { gemm_tile(g, blockIdx.x, blockIdx.y, blockIdx.z); }

// several small independent products in one launch: blockIdx.z selects the problem (batch = 1, no split-K)
constexpr int kMaxGroup = 12;
struct GemmGroupArgs { GemmKArgs g[kMaxGroup]; };
__global__ void __launch_bounds__(256) enf_gemm_group_kernel(const __grid_constant__ GemmGroupArgs G) {
  const GemmKArgs& g = G.g[blockIdx.z];
  if ((int)blockIdx.x * BM >= g.M || (int)blockIdx.y * BN >= g.N) return;
  gemm_tile(g, blockIdx.x, blockIdx.y, 0);
}

constexpr size_t kGemmSmem = (size_t)ST * BK * ((BM + 4) + (BN + 4)) * sizeof(float);
// the attribute is per DEVICE (and above the 48 KB default), so it is remembered per device ordinal, not per process
bool gemm_configure() {
  static bool done[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return false;
  if (dev >= 0 && dev < 64 && done[dev]) return true;
  const bool ok =
      cudaFuncSetAttribute(enf_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGemmSmem) == cudaSuccess &&
      cudaFuncSetAttribute(enf_gemm_group_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGemmSmem) == cudaSuccess;
  if (ok && dev >= 0 && dev < 64) done[dev] = true;
  return ok;
}

GemmKArgs pack_args(int M, int N, int K, EnfMat A, EnfMat B, EnfMat C, const EnfGemmOpts& o) {
  GemmKArgs g;
  g.A = A.p; g.sam = A.rs; g.sak = A.cs; g.sab = A.bs;
  g.B = B.p; g.sbk = B.rs; g.sbn = B.cs; g.sbb = B.bs;
  g.C = const_cast<float*>(C.p); g.scm = C.rs; g.scn = C.cs; g.scb = C.bs;
  g.bias = o.bias; g.bias_bs = o.bias_bs; g.aux = o.mul_gelu_grad; g.C2 = o.gelu_out; g.round_out = o.round_out;
  g.M = M; g.N = N; g.K = K; g.act_a = o.act_a; g.accumulate = o.accumulate; g.alpha = o.alpha;
  g.splitk = 1;
  g.kchunk = ((K + BK - 1) / BK) * BK;
  if (g.kchunk < BK) g.kchunk = BK;
  return g;
}

}  // namespace

bool enf_gemm_groupable(int M, int N, int K, const EnfGemmOpts& o) {
  return o.batch == 1 && !o.tc && K <= 1024 && (int64_t)((M + BM - 1) / BM) * ((N + BN - 1) / BN) <= 64;
}

int enf_gemm_group(cudaStream_t st, int n, const EnfGemmProblem* p) {
  if (n <= 0) return 0;
  if (!gemm_configure()) return -1;
  int launches = 0;
  for (int first = 0; first < n; first += kMaxGroup) {
    const int cnt = n - first < kMaxGroup ? n - first : kMaxGroup;
    GemmGroupArgs G;
    int gx = 1, gy = 1;
    for (int i = 0; i < cnt; ++i) {
      const EnfGemmProblem& q = p[first + i];
      G.g[i] = pack_args(q.M, q.N, q.K, q.A, q.B, q.C, q.o);
      const int tm = (q.M + BM - 1) / BM, tn = (q.N + BN - 1) / BN;
      if (tm > gx) gx = tm;
      if (tn > gy) gy = tn;
    }
    enf_gemm_group_kernel<<<dim3(gx, gy, cnt), 256, kGemmSmem, st>>>(G);
    ++launches;
  }
  return launches;
}

int enf_gemm(cudaStream_t st, int M, int N, int K, EnfMat A, EnfMat B, EnfMat C, const EnfGemmOpts& o) {
  if (M <= 0 || N <= 0 || o.batch <= 0) return 0;
  if (o.tc) {
    int r = enf_gemm_tc(st, M, N, K, A, B, C, o);
    if (r != 0) return r;
  }
  GemmKArgs g = pack_args(M, N, K, A, B, C, o);
  int tiles_m = (M + BM - 1) / BM, tiles_n = (N + BN - 1) / BN;
  int64_t tiles = (int64_t)tiles_m * tiles_n * o.batch;
  int splitk = 1;
  // split-K only when the result is accumulated atomically anyway and the grid would not fill the GPU
  if (o.accumulate && !o.mul_gelu_grad && tiles < 296 && K >= 512) {
    int want = (int)((592 + tiles - 1) / tiles);
    int maxs = (K + 127) / 128;
    splitk = want < maxs ? want : maxs;
    if (splitk < 1) splitk = 1;
  }
  int kchunk = (K + splitk - 1) / splitk;
  kchunk = ((kchunk + BK - 1) / BK) * BK;
  if (kchunk < BK) kchunk = BK;
  splitk = (K + kchunk - 1) / kchunk;
  if (splitk < 1) splitk = 1;
  g.splitk = splitk; g.kchunk = kchunk;
  dim3 grid(tiles_m, tiles_n, o.batch * splitk);
  if (!gemm_configure()) return -1;
  enf_gemm_kernel<<<grid, 256, kGemmSmem, st>>>(g);
  return 1;
}
