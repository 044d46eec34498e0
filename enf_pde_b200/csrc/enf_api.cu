// C ABI (include/enf_b200.h) and stage orchestration of the ENF cross-attention path.
//
//   W  fold weights            (A_q, c_q, W', b', W2g, b2g, M2g, c2g)
//   L  per-latent folds        (pose record Lam, ahat, k, v0, U, kappa, Weff, W3, b3)
//   X  per-query record xi
//   P  fused pair kernel       -> nbar, lse                    [the hot kernel]
//   Q  per-query tail          M2g, out_proj, block FFN, decode MLP -> out
// and the reverse of each for enf_xattn_bwd.  The algebra is tests/folded_model.py (validated on CPU
// against the unfused oracle); DESIGN.md lists every buffer.
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "enf_common.cuh"

namespace {

thread_local std::string g_err;
thread_local int g_launches = 0;

int fail(int code, const std::string& msg) { g_err = msg; return code; }

struct Buf { const char* name; size_t off; size_t n; };

struct Layout {
  std::vector<Buf> bufs;
  size_t total = 0;          // floats
  size_t acc_begin = 0, acc_end = 0;   // zeroed at the start of every bwd
  size_t add(const char* name, size_t n) {
    size_t off = total;
    bufs.push_back({name, off, n});
    total += (n + 63) & ~size_t(63);    // 256-byte granularity
    return off;
  }
  size_t off(const char* name) const {
    for (auto& b : bufs) if (!strcmp(b.name, name)) return b.off;
    return (size_t)-1;
  }
};

const char* kLeafNames[ENF_NUM_WEIGHT_LEAVES] = {
    "stem_w", "stem_b", "ln_attn_g", "ln_attn_b", "q_omega", "q_w1", "q_b1", "q_wf", "q_bf", "v_omega", "v_w1", "v_b1",
    "v_wf", "v_bf", "wq", "bq", "wk", "bk", "wv", "bv", "fv_w1", "fv_b1", "fv_g", "fv_beta", "fv_w2", "fv_b2", "mx_w1",
    "mx_b1", "mx_g", "mx_beta", "mx_w2", "mx_b2", "wo", "bo", "fb_w1", "fb_b1", "fb_g", "fb_beta", "fb_w2", "fb_b2",
    "m0_w", "m0_b", "m1_w", "m1_b", "m2_w", "m2_b"};

void leaf_sizes(const EnfDesc& D, int I, size_t* n) {
  const size_t d = D.d, H = D.H, L = D.L, O = D.O, Hd = H * d;
  size_t v[ENF_NUM_WEIGHT_LEAVES] = {
      L * d, d, d, d, I * (d / 2), d * d, d, d * d, d, I * (d / 2), d * d, d, d * d, d, d * Hd, Hd, d * Hd, Hd, d * Hd, Hd,
      d * d, d, d, d, d * 2 * Hd, 2 * Hd, d * d, d, d, d, d * d, d, Hd * Hd, Hd, Hd * Hd, Hd, Hd, Hd, Hd * Hd, Hd,
      Hd * d, d, d * d, d, d * O, O};
  if (D.flags & ENF_FLAG_NO_STEM) v[0] = v[1] = 0;
  if (D.flags & ENF_FLAG_SELF_BLOCK) {         // project_heads: out_proj (Hd, d); pointwise FFN d -> d -> d; no decode MLP
    v[32] = Hd * d; v[33] = d; v[34] = d * d; v[35] = d; v[36] = d; v[37] = d; v[38] = d * d; v[39] = d;
    for (int i = 40; i < ENF_NUM_WEIGHT_LEAVES; ++i) v[i] = 0;
  }
  memcpy(n, v, sizeof(v));
}

// the pair kernels' record layout; self-attention steps use get_sa_invariant's variant (Ponita2D: a third invariant)
EnfInvariantLayout record_layout(const EnfDesc& D) {
  EnfInvariantLayout r = enf_record_layout(D.invariant_kind, D.Dx, D.use_window);
  if ((D.flags & ENF_FLAG_SELF_BLOCK) && D.invariant_kind == ENF_INV_PONITA) {
    r.I = 3;
    if (r.win_kind == ENF_WIN_NP) r.win_row = r.I;
  }
  return r;
}
// tcgen05 pair kernels: tensor-core precision mode, a supported shape, and not a latent self-attention step
bool tc_fwd_on(const EnfDesc& D) {
  return D.precision == ENF_PREC_BF16 && enf_pairs_fwd_tc_supported(D.d, D.H) && !(D.flags & ENF_FLAG_SELF_BLOCK);
}

int validate(const EnfDesc* D, EnfInvariantLayout* rl) {
  if (!D) return fail(ENF_ERR_NULL_POINTER, "desc is NULL");
  if (D->B <= 0 || D->C <= 0 || D->Z <= 0 || D->L <= 0 || D->O <= 0) return fail(ENF_ERR_BAD_DESC, "B, C, Z, L, O must be positive");
  if (!(D->d == 16 || D->d == 32 || D->d == 64 || D->d == 128)) return fail(ENF_ERR_UNSUPPORTED, "num_hidden must be 16, 32, 64 or 128");
  if (D->H < 1 || D->H > 4) return fail(ENF_ERR_UNSUPPORTED, "num_heads must be 1..4");
  EnfInvariantLayout r = record_layout(*D);
  if (r.I < 0) return fail(ENF_ERR_BAD_DESC, "unknown invariant_kind");
  int k = D->invariant_kind;
  bool dx_ok = (k <= ENF_INV_ABS_POS) ? (D->Dx >= 1 && D->Dx <= 3)
               : (k == ENF_INV_BALL || k == ENF_INV_BALL_LAT) ? (D->Dx == 3) : (D->Dx == 2);
  if (!dx_ok) return fail(ENF_ERR_BAD_DESC, "num_in (Dx) does not match the invariant (rel/norm/abs: 1..3, ball*: 3, others: 2)");
  if ((int64_t)D->B * D->Z * D->H > 65535) return fail(ENF_ERR_UNSUPPORTED, "B*Z*H must be <= 65535 per call (shard the fields)");
  if (D->B > 65535) return fail(ENF_ERR_UNSUPPORTED, "B must be <= 65535");
  if (D->precision != ENF_PREC_FP32 && D->precision != ENF_PREC_BF16) return fail(ENF_ERR_BAD_DESC, "unknown precision");
  if (D->flags & ~(ENF_FLAG_FORWARD_ONLY | ENF_FLAG_RECOMPUTE | ENF_FLAG_OUT_BF16 | ENF_FLAG_FROZEN_RELU | ENF_FLAG_SELF_BLOCK | ENF_FLAG_NO_STEM |
                   ENF_FLAG_GRAD_X))
    return fail(ENF_ERR_BAD_DESC, "unknown bits in flags");
  if ((D->flags & ENF_FLAG_GRAD_X) && (D->flags & (ENF_FLAG_FORWARD_ONLY | ENF_FLAG_SELF_BLOCK)))
    return fail(ENF_ERR_BAD_DESC, "ENF_FLAG_GRAD_X needs a backward (not ENF_FLAG_FORWARD_ONLY) of a decode call (not ENF_FLAG_SELF_BLOCK)");
  if ((D->flags & ENF_FLAG_NO_STEM) && D->L != D->d) return fail(ENF_ERR_BAD_DESC, "ENF_FLAG_NO_STEM: a is the hidden state, L must equal d");
  if (D->flags & ENF_FLAG_SELF_BLOCK) {
    if (D->C != D->Z || D->O != D->d) return fail(ENF_ERR_BAD_DESC, "ENF_FLAG_SELF_BLOCK: the queries are the latents (C == Z) and out is the hidden state (O == d)");
    if (D->flags & (ENF_FLAG_RECOMPUTE | ENF_FLAG_OUT_BF16 | ENF_FLAG_FROZEN_RELU))
      return fail(ENF_ERR_UNSUPPORTED, "ENF_FLAG_SELF_BLOCK does not combine with RECOMPUTE / OUT_BF16 / FROZEN_RELU");
  }
  if ((D->flags & ENF_FLAG_OUT_BF16) && (!(D->flags & ENF_FLAG_FORWARD_ONLY) || !enf_thin_supported(D->d, D->O)))
    return fail(ENF_ERR_UNSUPPORTED, "ENF_FLAG_OUT_BF16 needs ENF_FLAG_FORWARD_ONLY and num_out <= 4");
  if ((D->flags & ENF_FLAG_FROZEN_RELU) && D->precision != ENF_PREC_FP32)
    return fail(ENF_ERR_UNSUPPORTED, "ENF_FLAG_FROZEN_RELU is implemented by the fp32 kernels only");
  if (D->chunk_fields < 0 || D->reserved[0] || D->reserved[1] || D->reserved[2])
    return fail(ENF_ERR_BAD_DESC, "chunk_fields must be >= 0 and the reserved fields 0");
  if (rl) *rl = r;
  return ENF_OK;
}

// tensor-core backward wherever the tensor-core forward runs (d in {32, 64, 128}, H <= 4; more than two heads at d >= 64, and
// four at d = 32, run as head groups of <= 2): a backward on the fp32 kernels behind a
// 16-bit-operand forward mixes two different roundings of the same activations (measured: 2e-2 on single weight-gradient leaves)
bool use_tc_bwd(const EnfDesc& D) { return tc_fwd_on(D) && enf_pairs_bwd_tc_supported(D.d, D.H); }

// fields per backward chunk: everything O(B*C*Z) that only lives between the pair kernels of one chunk is sized by this.
// Default (stash) mode: one chunk = the whole batch.
int chunk_fields(const EnfDesc& D) {
  if (!(D.flags & ENF_FLAG_RECOMPUTE) || !use_tc_bwd(D)) return D.B;
  int n = D.chunk_fields > 0 ? D.chunk_fields : 4;
  return n < D.B ? n : D.B;
}

Layout make_layout(const EnfDesc& D, const EnfRecordLayout& rl) {
  Layout Y;
  const bool train = !(D.flags & ENF_FLAG_FORWARD_ONLY);      // forward only: no backward state, no gradient buffers
  const size_t d = D.d, H = D.H, Hd = H * d, d2 = d * d;
  const size_t BZ = (size_t)D.B * D.Z, BC = (size_t)D.B * D.C;
  Y.add("A_q", d * Hd); Y.add("c_q", Hd); Y.add("Wp", d2); Y.add("bp", d); Y.add("W2g", d * 2 * Hd); Y.add("b2g", 2 * Hd);
  Y.add("M2g", d2); Y.add("c2g", d); Y.add("P1", Hd * Hd); Y.add("b1", Hd); Y.add("W_A", Hd * Hd); Y.add("b_A", Hd);
  Y.add("dP1", Hd * Hd); Y.add("db1", Hd); Y.add("q_w1T", d2); Y.add("v_w1T", d2); Y.add("WpT", d2);
  Y.add("lam", BZ * ENF_LAM_SIZE);
  if (D.flags & ENF_FLAG_FROZEN_RELU) Y.add("lam_mask", BZ * ENF_LAM_SIZE);
  Y.add("a0", BZ * d); Y.add("acore", BZ * d); Y.add("arstd", BZ); Y.add("ahat", BZ * d);
  Y.add("k", BZ * Hd); Y.add("v0", BZ * Hd); Y.add("U", BZ * Hd); Y.add("kappa", BZ * H);
  Y.add("Weff", BZ * H * d2); Y.add("beff", BZ * Hd); Y.add("W3", BZ * H * d2); Y.add("b3", BZ * Hd);
  {
    // transposed W3 copies: only the fp32-FMA backward reads them
    const bool tc_both = use_tc_bwd(D);
    // ... and, there, the cotangent of Weff gets a buffer of its own (the tensor-core backward never reads the fp32 W3
    // again, so it reuses that one): a backward leaves the forward state intact and can be repeated
    if (train && !tc_both) { Y.add("W3T", BZ * H * d2); Y.add("dWeff", BZ * H * d2); }
  }
  if (tc_fwd_on(D)) {
    // operand images: rows of max(d, 64) 16-bit features (d = 32 keeps the 128-byte row pitch), counted in floats
    const size_t dimg = d * (d < 64 ? 64 : d) / 2;
    Y.add("img_q_w1", dimg); Y.add("img_v_w1", dimg); Y.add("img_Wp", dimg); Y.add("img_W3", BZ * H * dimg);
    if (train) Y.add("slog", BC * (size_t)D.Z * H);
    // tf32 stage GEMMs: activated copies of the decode-MLP pre-activations (their A operands arrive by TMA) and the
    // low parts W - trunc_tf32(W) of the weights those GEMMs multiply by (3-term split product)
    Y.add("fo_act", BC * Hd); Y.add("o1_act", BC * d); Y.add("o2_act", BC * d);
    Y.add("lo_W_A", Hd * Hd); Y.add("lo_fb_w2", Hd * Hd); Y.add("lo_m0_w", Hd * d); Y.add("lo_m1_w", d2); Y.add("lo_mx_w1", d2);
    if (train && use_tc_bwd(D)) {
      Y.add("img_q_w1_lo", dimg); Y.add("img_v_w1_lo", dimg);
      const size_t Cpad = (size_t)((D.C + 127) / 128) * 128;      // kernels A / B work on whole 128-query tiles
      // per-(query, latent) tensors that live between the pair kernels of ONE backward chunk: all fields in the default
      // (stash) mode, chunk_fields fields with ENF_FLAG_RECOMPUTE
      const size_t cZ = (size_t)chunk_fields(D) * D.Z, cC = (size_t)chunk_fields(D) * D.C;
      Y.add("dthat", cZ * Cpad * d / 2); Y.add("ds_tc", cC * (size_t)D.Z * H); Y.add("Dg", BC * H);
      Y.add("dnb16", (size_t)D.B * Cpad * Hd / 2);
      Y.add("duv", cC * (size_t)D.Z * 8);
      // fp16 operand images of `that` per (field, latent, 128-query tile), stashed by the forward for backward kernel A
      Y.add("that_img", cZ * Cpad * (d < 64 ? 64 : d) / 2);
      // rstd * gelu' of the same layer (fp16), stashed for backward kernel B: with `that` it is all the LayerNorm / gelu backward needs
      Y.add("dgr", cZ * Cpad * d / 2); Y.add("trstd", cZ * Cpad);
    }
  }
  Y.add("xi", BC * ENF_F_XI);
  Y.add("nbar", BC * Hd); Y.add("lse", BC * H);
  Y.add("e1", BC * Hd); Y.add("e3c", BC * Hd); Y.add("erstd", BC); Y.add("e3", BC * Hd);
  Y.add("fo", BC * Hd); Y.add("o1p", BC * d); Y.add("o2p", BC * d);
  if (!train) return Y;
  Y.add("s0", BC * Hd); Y.add("s1", BC * Hd); Y.add("d_o2p", BC * d); Y.add("d_o1p", BC * d);
  Y.add("dbeff", BZ * Hd); Y.add("dk", BZ * Hd); Y.add("dv0", BZ * Hd); Y.add("dahat", BZ * d); Y.add("da0", BZ * d);
  if (D.flags & ENF_FLAG_SELF_BLOCK) { Y.add("da0x", BZ * d); Y.add("g_xi", BC * ENF_F_XI); }
  // ---- accumulators, zeroed at the start of each bwd ----
  Y.acc_begin = Y.total;
  Y.add("g_W3", BZ * H * d2); Y.add("g_b3", BZ * Hd); Y.add("g_U", BZ * Hd); Y.add("g_kappa", BZ * H);
  Y.add("g_lam", BZ * ENF_LAM_SIZE); Y.add("g_sigma", BZ); Y.add("gmax", 64);
  Y.add("gf_A_q", d * Hd); Y.add("gf_c_q", Hd); Y.add("gf_Wp", d2); Y.add("gf_bp", d); Y.add("gf_W2g", d * 2 * Hd);
  Y.add("gf_b2g", 2 * Hd); Y.add("gf_M2g", d2); Y.add("gf_c2g", d); Y.add("gf_W_A", Hd * Hd); Y.add("gf_b_A", Hd);
  size_t n[ENF_NUM_WEIGHT_LEAVES];
  leaf_sizes(D, rl.I, n);
  static const std::vector<std::string> names = [] {
    std::vector<std::string> v;
    for (int i = 0; i < ENF_NUM_WEIGHT_LEAVES; ++i) v.push_back(std::string("gw_") + kLeafNames[i]);
    return v;
  }();
  for (int i = 0; i < ENF_NUM_WEIGHT_LEAVES; ++i) Y.add(names[i].c_str(), n[i]);
  if (D.flags & ENF_FLAG_GRAD_X) Y.add("g_xi", BC * ENF_F_XI);     // cotangent of the query records (reduced over latents)
  Y.acc_end = Y.total;
  return Y;
}

std::mutex g_mu;
struct FwdState { EnfDesc D; int64_t xbs; };
std::map<void*, FwdState> g_fwd_state;    // workspaces that currently hold a forward (erased by enf_workspace_release)

// optional live timing of the two fused pair kernels (bench.py's roofline line): a ring of CUDA event
// pairs per kernel, recorded on the call's stream; enf_profile_collect drains it.
constexpr int kProfRing = 256;
bool g_prof_on = false;
cudaEvent_t g_prof_ev[2][kProfRing][2];
int g_prof_dev[2][kProfRing];             // device the slot's events were created on (-1: none); events are per device
bool g_prof_init = false;
long g_prof_count[2] = {0, 0};
void prof_mark(int which, int edge, cudaStream_t st) {
  if (!g_prof_on) return;
  if (!g_prof_init) {
    for (int w = 0; w < 2; ++w) for (int i = 0; i < kProfRing; ++i) g_prof_dev[w][i] = -1;
    g_prof_init = true;
  }
  int slot = (int)(g_prof_count[which] % kProfRing);
  int dev = 0;
  cudaGetDevice(&dev);
  if (g_prof_dev[which][slot] != dev) {
    if (g_prof_dev[which][slot] >= 0) { cudaEventDestroy(g_prof_ev[which][slot][0]); cudaEventDestroy(g_prof_ev[which][slot][1]); }
    cudaEventCreate(&g_prof_ev[which][slot][0]);
    cudaEventCreate(&g_prof_ev[which][slot][1]);
    g_prof_dev[which][slot] = dev;
  }
  cudaEventRecord(g_prof_ev[which][slot][edge], st);
  if (edge == 1) g_prof_count[which]++;
}

struct LeafCopy { const float* src[ENF_NUM_WEIGHT_LEAVES]; float* dst[ENF_NUM_WEIGHT_LEAVES]; int n[ENF_NUM_WEIGHT_LEAVES]; };
__global__ void copy_leaves_kernel(LeafCopy t) {
  const int leaf = blockIdx.y;
  float* dst = t.dst[leaf];
  if (!dst) return;
  const float* src = t.src[leaf];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < t.n[leaf]; i += gridDim.x * blockDim.x) dst[i] = src[i];
}

struct Ctx {
  cudaStream_t st;
  float* ws;
  const Layout* Y;
  int launches = 0;
  bool tc = false;           // tensor-core precision mode: big stage GEMMs run on the tf32 kernels
  bool gemm_failed = false;
  float* f(const char* name) const { return ws + Y->off(name); }
  // Products issued between begin_group() / end_group() must be mutually independent (no one reads or non-atomically
  // rewrites another's output): the small ones are collected and go out in ONE launch (their time is launch + pipeline
  // latency, not flops), the others launch immediately.
  bool grouping = false;
  std::vector<EnfGemmProblem> pending;
  void begin_group() { grouping = true; }
  void end_group() {
    grouping = false;
    if (pending.empty()) return;
    int r = enf_gemm_group(st, (int)pending.size(), pending.data());
    if (r < 0) gemm_failed = true; else launches += r;
    pending.clear();
  }
  void gemm(int M, int N, int K, EnfMat A, EnfMat B, EnfMat C, const EnfGemmOpts& o = EnfGemmOpts()) {
    EnfGemmOpts oo = o;
    if (!tc) oo.tc = 0;       // callers mark the big tail / W3 products (with_lo, opt_acc_big); honoured in tensor-core mode only
    if (M <= 0 || N <= 0) return;
    if (grouping && enf_gemm_groupable(M, N, K, oo)) { pending.push_back(EnfGemmProblem{M, N, K, A, B, C, oo}); return; }
    int r = enf_gemm(st, M, N, K, A, B, C, oo);
    if (r < 0) gemm_failed = true; else launches += r;
  }
};

EnfGemmOpts opt_bias(const float* bias) { EnfGemmOpts o; o.bias = bias; return o; }
// big-M product by a small weight: tf32 3-term split kernel when the weight's low part is available
EnfGemmOpts with_lo(EnfGemmOpts o, const float* b_lo) { o.b_lo = b_lo; o.tc = b_lo ? 1 : 0; return o; }
// weight gradient reduced over all queries / all W3 rows: tf32 kernel in tensor-core mode
EnfGemmOpts opt_acc_big() { EnfGemmOpts o; o.accumulate = 1; o.tc = 1; return o; }
EnfGemmOpts opt_acc() { EnfGemmOpts o; o.accumulate = 1; return o; }

EnfPairParams pair_params(const EnfDesc& D, const EnfRecordLayout& rl, const EnfWeights& w, const Ctx& c,
                          const float* sigma, int64_t xi_bs) {
  EnfPairParams p;
  memset(&p, 0, sizeof(p));
  p.B = D.B; p.C = D.C; p.Z = D.Z; p.H = D.H; p.rec = rl;
  p.xi = c.f("xi"); p.xi_bs = xi_bs; p.lam = c.f("lam"); p.sigma = sigma;
  p.lam_mask = (D.flags & ENF_FLAG_FROZEN_RELU) ? c.f("lam_mask") : nullptr;
  p.q_omega = w.q_omega; p.v_omega = w.v_omega;
  p.q_w1 = w.q_w1; p.q_b1 = w.q_b1; p.v_w1 = w.v_w1; p.v_b1 = w.v_b1;
  p.Wp = c.f("Wp"); p.bp = c.f("bp");
  p.U = c.f("U"); p.kappa = c.f("kappa"); p.W3 = c.f("W3"); p.b3 = c.f("b3");
  p.nbar = c.f("nbar"); p.lse = c.f("lse");
  return p;
}

bool check_weights(const EnfDesc& D, const EnfWeights* w);

// parameters of the tensor-core pair forward; `stash`: also write the backward's operand stash (that_img / dgr / trstd)
EnfPairTcParams tc_fwd_params(const EnfDesc& D, const EnfRecordLayout& rl, const EnfWeights& w, const Ctx& c, const EnfPairParams& pp,
                              bool keep_logits, bool stash) {
  EnfPairTcParams tp;
  memset(&tp, 0, sizeof(tp));
  tp.B = D.B; tp.C = D.C; tp.Z = D.Z; tp.rec = rl;
  tp.xi = pp.xi; tp.xi_bs = pp.xi_bs; tp.lam = pp.lam; tp.sigma = pp.sigma;
  tp.q_omega = w.q_omega; tp.v_omega = w.v_omega; tp.q_b1 = w.q_b1; tp.v_b1 = w.v_b1; tp.bp = c.f("bp");
  tp.img_q_w1 = (const uint8_t*)c.f("img_q_w1"); tp.img_v_w1 = (const uint8_t*)c.f("img_v_w1");
  tp.img_Wp = (const uint8_t*)c.f("img_Wp"); tp.img_W3 = (const uint8_t*)c.f("img_W3");
  tp.U = pp.U; tp.kappa = pp.kappa; tp.b3 = pp.b3; tp.nbar = pp.nbar; tp.lse = pp.lse; tp.slog = keep_logits ? c.f("slog") : nullptr;
  tp.that_img = stash ? reinterpret_cast<uint8_t*>(c.f("that_img")) : nullptr;
  tp.dgr = stash ? reinterpret_cast<uint4*>(c.f("dgr")) : nullptr;
  tp.trstd = stash ? c.f("trstd") : nullptr;
  return tp;
}
// restrict a pair-forward launch to the fields [b0, b0 + nb): every per-field / per-latent pointer moves; the operand stash
// is chunk-local (it always starts at its buffer's base)
void shift_fields(EnfPairTcParams& tp, const EnfDesc& D, int b0, int nb) {
  const int64_t bz = (int64_t)b0 * D.Z, bc = (int64_t)b0 * D.C, Hd = (int64_t)D.H * D.d;
  tp.B = nb;
  tp.xi += b0 * tp.xi_bs; tp.lam += bz * ENF_LAM_SIZE; if (tp.sigma) tp.sigma += bz;
  tp.img_W3 += bz * D.H * (int64_t)D.d * (D.d < 64 ? 64 : D.d) * 2;
  tp.U += bz * Hd; tp.kappa += bz * D.H; tp.b3 += bz * Hd; tp.nbar += bc * Hd; tp.lse += bc * D.H;
  if (tp.slog) tp.slog += bz * D.C * D.H;
}
// same for the pair backward: the A -> B -> C hand-over tensors (dthat, ds, duv) and the stash are chunk-local
void shift_fields(EnfPairTcBwdParams& tp, const EnfDesc& D, int b0, int nb) {
  const int64_t bz = (int64_t)b0 * D.Z, bc = (int64_t)b0 * D.C, Hd = (int64_t)D.H * D.d;
  const int64_t ntiles = (D.C + 127) / 128;
  tp.B = nb;
  tp.xi += b0 * tp.xi_bs; tp.lam += bz * ENF_LAM_SIZE; if (tp.sigma) tp.sigma += bz;
  tp.img_W3 += bz * D.H * (int64_t)D.d * (D.d < 64 ? 64 : D.d) * 2;
  tp.U += bz * Hd; tp.b3 += bz * Hd; tp.slog += bz * D.C * D.H; tp.lse += bc * D.H; tp.nbar += bc * Hd;
  tp.dnbar += bc * Hd; tp.Dg += bc * D.H; tp.dnb16 += (int64_t)b0 * ntiles * 128 * Hd / 8;
  tp.g_W3 += bz * D.H * (int64_t)D.d * D.d; tp.g_b3 += bz * Hd;
  tp.g_U += bz * Hd; tp.g_kappa += bz * D.H; tp.g_lam += bz * ENF_LAM_SIZE; tp.g_sigma += bz;
  if (tp.g_xi) tp.g_xi += bc * ENF_F_XI;
}

// argument checks shared by enf_xattn_fwd and enf_xattn_bwd
int check_call(const EnfDesc& D, const EnfWeights* w, const float* x, int64_t x_batch_stride, const float* p, const float* a,
               const float* sigma, void* workspace) {
  const bool self = (D.flags & ENF_FLAG_SELF_BLOCK) != 0;
  if (!w || (!x && !self) || !p || !a || !workspace) return fail(ENF_ERR_NULL_POINTER, "NULL argument");
  if (!check_weights(D, w)) return fail(ENF_ERR_NULL_POINTER, "EnfWeights has a NULL leaf");
  if (D.use_window && !sigma) return fail(ENF_ERR_NULL_POINTER, "sigma is NULL but use_window is set (the reference asserts the same)");
  if (!self && x_batch_stride != 0 && x_batch_stride != (int64_t)D.C * D.Dx) return fail(ENF_ERR_BAD_DESC, "x_batch_stride must be 0 or C*Dx");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return fail(ENF_ERR_NO_DEVICE, "no CUDA device (there is no CPU fallback)"); }
  if (reinterpret_cast<uintptr_t>(workspace) & 255) return fail(ENF_ERR_WORKSPACE, "workspace must be 256-byte aligned");
  return ENF_OK;
}

bool check_weights(const EnfDesc& D, const EnfWeights* w) {
  const float* const* p = reinterpret_cast<const float* const*>(w);
  size_t n[ENF_NUM_WEIGHT_LEAVES];
  leaf_sizes(D, 1, n);
  for (int i = 0; i < ENF_NUM_WEIGHT_LEAVES; ++i) if (!p[i] && n[i]) return false;      // leaves the call does not use may be NULL
  return true;
}

}  // namespace

extern "C" {

int enf_abi_version(void) { return ENF_B200_ABI_VERSION; }

int enf_invariant_dim(int kind, int Dx) { return enf_record_layout(kind, Dx, 1).I; }
int enf_pose_dim(int kind, int Dx) { return enf_record_layout(kind, Dx, 1).P; }

const char* enf_last_error(void) { return g_err.c_str(); }

int enf_profile_enable(int on) {
  g_prof_on = on != 0;
  g_prof_count[0] = g_prof_count[1] = 0;
  return 0;
}
int enf_profile_collect(int which, float* ms_out, int max_out) {
  if (which < 0 || which > 1 || !ms_out) return -1;
  long n = g_prof_count[which];
  if (n > kProfRing) n = kProfRing;
  if (n > max_out) n = max_out;
  long first = g_prof_count[which] - n;
  for (long i = 0; i < n; ++i) {
    int slot = (int)((first + i) % kProfRing);
    float ms = -1.f;
    if (cudaEventSynchronize(g_prof_ev[which][slot][1]) != cudaSuccess) return -1;
    if (cudaEventElapsedTime(&ms, g_prof_ev[which][slot][0], g_prof_ev[which][slot][1]) != cudaSuccess) return -1;
    ms_out[i] = ms;
  }
  g_prof_count[which] = 0;
  return (int)n;
}

int enf_last_launch_count(void) { return g_launches; }
}  // extern "C"
// shared by the other translation units behind the same ABI (enf_ode.cu): thread-local message of enf_last_error()
int enf_set_error(int code, const char* msg) { return fail(code, msg ? msg : ""); }
extern "C" {

int enf_debug_gemm(int use_tc, int M, int N, int K, const float* A, int64_t a_rs, int64_t a_cs, const float* B, int64_t b_rs,
                   int64_t b_cs, const float* B_lo, float* C, int64_t c_rs, const float* bias, const float* aux, float* gelu_out,
                   int accumulate, enf_stream_t stream) {
  if (!A || !B || !C) return fail(ENF_ERR_NULL_POINTER, "NULL argument");
  EnfGemmOpts o;
  o.b_lo = B_lo;
  o.bias = bias; o.mul_gelu_grad = aux; o.gelu_out = gelu_out; o.accumulate = accumulate; o.tc = use_tc;
  int r = enf_gemm((cudaStream_t)stream, M, N, K, enf_mat(A, a_rs, a_cs), enf_mat(B, b_rs, b_cs), enf_mat(C, c_rs), o);
  if (r < 0) return fail(ENF_ERR_CUDA, "GEMM could not be configured");
  return r;
}

size_t enf_xattn_workspace_bytes(const EnfDesc* desc) {
  EnfInvariantLayout rl;
  if (validate(desc, &rl) != ENF_OK) return 0;
  return make_layout(*desc, rl).total * sizeof(float);
}

int enf_xattn_chunk_for_cap(const EnfDesc* desc, size_t cap_bytes) {
  EnfInvariantLayout rl;
  if (validate(desc, &rl) != ENF_OK) return 0;
  EnfDesc D = *desc;
  D.flags |= ENF_FLAG_RECOMPUTE;
  int lo = 0, hi = D.B;                     // the workspace grows monotonically with chunk_fields: bisect
  while (lo < hi) {
    const int mid = (lo + hi + 1) / 2;
    D.chunk_fields = mid;
    if (make_layout(D, rl).total * sizeof(float) <= cap_bytes) lo = mid; else hi = mid - 1;
  }
  return lo;
}

int enf_xattn_dispatch(const EnfDesc* desc, int* fwd_tc, int* bwd_tc) {
  int rc = validate(desc, nullptr);
  if (rc != ENF_OK) return rc;
  const bool f = tc_fwd_on(*desc);
  if (fwd_tc) *fwd_tc = f ? 1 : 0;
  if (bwd_tc) *bwd_tc = (f && use_tc_bwd(*desc) && !(desc->flags & ENF_FLAG_FORWARD_ONLY)) ? 1 : 0;
  return ENF_OK;
}

void enf_workspace_release(void* workspace) {
  std::lock_guard<std::mutex> lk(g_mu);
  g_fwd_state.erase(workspace);
}

int64_t enf_debug_ws_offset(const EnfDesc* desc, const char* name, int64_t* num_floats) {
  EnfInvariantLayout rl;
  if (validate(desc, &rl) != ENF_OK || !name) return -1;
  Layout Y = make_layout(*desc, rl);
  for (auto& b : Y.bufs)
    if (!strcmp(b.name, name)) { if (num_floats) *num_floats = (int64_t)b.n; return (int64_t)(b.off * sizeof(float)); }
  return -1;
}

int enf_xattn_fwd(const EnfDesc* desc, const EnfWeights* w, const float* x, int64_t x_batch_stride, const float* p,
                  const float* a, const float* sigma, float* out, void* workspace, size_t workspace_bytes,
                  enf_stream_t stream) {
  g_launches = 0;
  EnfInvariantLayout rl;
  int rc = validate(desc, &rl);
  if (rc != ENF_OK) return rc;
  const EnfDesc& D = *desc;
  if (!out) return fail(ENF_ERR_NULL_POINTER, "NULL argument");
  if ((rc = check_call(D, w, x, x_batch_stride, p, a, sigma, workspace)) != ENF_OK) return rc;
  const bool use_tc = tc_fwd_on(D);   // other shapes (and latent self-attention steps): fp32 kernels
  const bool train = !(D.flags & ENF_FLAG_FORWARD_ONLY);
  const bool self = (D.flags & ENF_FLAG_SELF_BLOCK) != 0, no_stem = (D.flags & ENF_FLAG_NO_STEM) != 0;
  Layout Y = make_layout(D, rl);
  if (workspace_bytes < Y.total * sizeof(float)) return fail(ENF_ERR_WORKSPACE, "workspace too small: see enf_xattn_workspace_bytes");

  Ctx c; c.st = (cudaStream_t)stream; c.ws = (float*)workspace; c.Y = &Y; c.tc = use_tc;
  cudaStream_t st = c.st;
  const int d = D.d, H = D.H, Hd = H * d, L = D.L, O = D.O;
  const int64_t BZ = (int64_t)D.B * D.Z, BC = (int64_t)D.B * D.C;
  const int Bx = (x_batch_stride == 0 && !self) ? 1 : D.B;
  // ---- W: fold weights --------------------------------------------------------------------------
  c.begin_group();
  c.gemm(d, Hd, d, enf_mat(w->q_wf, d), enf_mat(w->wq, Hd), enf_mat(c.f("A_q"), Hd));
  c.gemm(1, Hd, d, enf_mat(w->q_bf, d), enf_mat(w->wq, Hd), enf_mat(c.f("c_q"), Hd), opt_bias(w->bq));
  c.gemm(d, d, d, enf_mat(w->v_wf, d), enf_mat(w->fv_w1, d), enf_mat(c.f("Wp"), d));
  c.gemm(1, d, d, enf_mat(w->v_bf, d), enf_mat(w->fv_w1, d), enf_mat(c.f("bp"), d), opt_bias(w->fv_b1));
  c.launches += enf_launch_rowscale(st, w->fv_w2, w->fv_g, c.f("W2g"), d, 2 * Hd);
  c.gemm(1, 2 * Hd, d, enf_mat(w->fv_beta, d), enf_mat(w->fv_w2, 2 * Hd), enf_mat(c.f("b2g"), 2 * Hd), opt_bias(w->fv_b2));
  c.launches += enf_launch_rowscale(st, w->mx_w2, w->mx_g, c.f("M2g"), d, d);
  c.gemm(1, d, d, enf_mat(w->mx_beta, d), enf_mat(w->mx_w2, d), enf_mat(c.f("c2g"), d), opt_bias(w->mx_b2));
  c.end_group();
  // tail fold (exact algebra, tests/folded_model.py): mixer Dense_1, out_proj and the block FFN's Dense_0 are three
  // linear maps in a row:  e1 = nbar W_A + b_A,  W_A = blockdiag(M2g) wo fb_w1,  b_A = (tile(c2g) wo + bo) fb_w1 + fb_b1
  if (self) {
    // latent self-attention step (project_heads, residual): mixer Dense_1 and out_proj fold into  y = nbar P1 + b1,
    // P1 = blockdiag(M2g) wo (Hd, d),  b1 = tile(c2g) wo + bo (d); the residual sits between this and the FFN
    EnfGemmOpts ob; ob.batch = H;
    c.gemm(d, d, d, enf_mat(c.f("M2g"), d), enf_mat(w->wo, d, 1, (int64_t)d * d), enf_mat(c.f("P1"), d, 1, (int64_t)d * d), ob);
    if (cudaMemcpyAsync(c.f("b1"), w->bo, d * sizeof(float), cudaMemcpyDeviceToDevice, st) != cudaSuccess)
      return fail(ENF_ERR_CUDA, "copy of out_proj bias failed");
    for (int h = 0; h < H; ++h)
      c.gemm(1, d, d, enf_mat(c.f("c2g"), d), enf_mat(w->wo + (int64_t)h * d * d, d), enf_mat(c.f("b1"), d), opt_acc());
  } else {
    EnfGemmOpts ob; ob.batch = H;
    c.gemm(d, Hd, d, enf_mat(c.f("M2g"), d), enf_mat(w->wo, Hd, 1, (int64_t)d * Hd), enf_mat(c.f("P1"), Hd, 1, (int64_t)d * Hd), ob);
    if (cudaMemcpyAsync(c.f("b1"), w->bo, Hd * sizeof(float), cudaMemcpyDeviceToDevice, st) != cudaSuccess)
      return fail(ENF_ERR_CUDA, "copy of out_proj bias failed");
    for (int h = 0; h < H; ++h)      // head by head in stream order: a deterministic sum
      c.gemm(1, Hd, d, enf_mat(c.f("c2g"), d), enf_mat(w->wo + (int64_t)h * d * Hd, Hd), enf_mat(c.f("b1"), Hd), opt_acc());
    c.begin_group();
    c.gemm(Hd, Hd, Hd, enf_mat(c.f("P1"), Hd), enf_mat(w->fb_w1, Hd), enf_mat(c.f("W_A"), Hd));
    c.gemm(1, Hd, Hd, enf_mat(c.f("b1"), Hd), enf_mat(w->fb_w1, Hd), enf_mat(c.f("b_A"), Hd), opt_bias(w->fb_b1));
    c.end_group();
  }
  if (use_tc) {
    EnfSplitList sl;
    const float* src[5] = {c.f("W_A"), w->fb_w2, w->m0_w, w->m1_w, w->mx_w1};
    float* dst[5] = {c.f("lo_W_A"), c.f("lo_fb_w2"), c.f("lo_m0_w"), c.f("lo_m1_w"), c.f("lo_mx_w1")};
    const int nn[5] = {Hd * Hd, Hd * Hd, Hd * d, d * d, d * d};
    for (int i = 0; i < 5; ++i) { sl.src[i] = src[i]; sl.dst[i] = dst[i]; sl.n[i] = nn[i]; }
    sl.count = 5;
    c.launches += enf_launch_split_lo(st, sl);
  }

  // ---- L: per-latent folds ----------------------------------------------------------------------
  if (self) c.launches += enf_launch_pose_record(st, D.invariant_kind, D.Dx, rl.P, rl.I, BZ, p, c.f("lam"));
  else c.launches += enf_launch_latent_record(st, D, p, c.f("lam"));
  if (D.flags & ENF_FLAG_FROZEN_RELU)      // second pose set: the relu pattern's expansion point
    c.launches += enf_launch_latent_record(st, D, p + BZ * rl.P, c.f("lam_mask"));
  if (no_stem) {
    if (cudaMemcpyAsync(c.f("a0"), a, BZ * d * sizeof(float), cudaMemcpyDeviceToDevice, st) != cudaSuccess)
      return fail(ENF_ERR_CUDA, "copy of the hidden latent state failed");
  } else {
    c.gemm((int)BZ, d, L, enf_mat(a, L), enf_mat(w->stem_w, d), enf_mat(c.f("a0"), d), opt_bias(w->stem_b));
  }
  c.launches += enf_launch_ln_fwd(st, c.f("a0"), BZ, d, w->ln_attn_g, w->ln_attn_b, c.f("acore"), c.f("ahat"), c.f("arstd"), 0);
  c.begin_group();
  c.gemm((int)BZ, Hd, d, enf_mat(c.f("ahat"), d), enf_mat(w->wk, Hd), enf_mat(c.f("k"), Hd), opt_bias(w->bk));
  c.gemm((int)BZ, Hd, d, enf_mat(c.f("ahat"), d), enf_mat(w->wv, Hd), enf_mat(c.f("v0"), Hd), opt_bias(w->bv));
  c.end_group();
  {
    EnfGemmOpts o; o.batch = H;     // U[bz,h,i] = sum_j A_q[i, h*d+j] k[bz,h,j]
    c.gemm((int)BZ, d, d, enf_mat(c.f("k"), Hd, 1, d), enf_mat(c.f("A_q"), 1, Hd, d), enf_mat(c.f("U"), Hd, 1, d), o);
    // kappa[bz,h] = sum_j c_q[h*d+j] k[bz,h,j]
    c.gemm((int)BZ, 1, d, enf_mat(c.f("k"), Hd, 1, d), enf_mat(c.f("c_q"), 1, 0, d), enf_mat(c.f("kappa"), H, 1, 1), o);
  }
  c.launches += enf_launch_weff(st, D, c.f("W2g"), c.f("b2g"), c.f("v0"), c.f("Weff"), c.f("beff"));
  c.gemm((int)(BZ * H * d), d, d, enf_mat(c.f("Weff"), d), enf_mat(w->mx_w1, d), enf_mat(c.f("W3"), d),
         with_lo(EnfGemmOpts(), use_tc ? c.f("lo_mx_w1") : nullptr));
  c.gemm((int)(BZ * H), d, d, enf_mat(c.f("beff"), d), enf_mat(w->mx_w1, d), enf_mat(c.f("b3"), d), opt_bias(w->mx_b1));

  // ---- X, P ---------------------------------------------------------------------------------------
  if (self) c.launches += enf_launch_pose_features(st, D.invariant_kind, D.Dx, rl.P, BZ, p, c.f("xi"));      // x = p
  else c.launches += enf_launch_query_features(st, D, x, x_batch_stride, Bx, c.f("xi"));
  EnfPairParams pp = pair_params(D, rl, *w, c, D.use_window ? sigma : nullptr, Bx == 1 ? 0 : (int64_t)D.C * ENF_F_XI);
  int nl;
  if (use_tc) {
    // operand images: bf16, pre-swizzled, of the TRANSPOSED weights ([out][in]) = K-major B tiles
    c.launches += enf_launch_transpose(st, w->q_w1, c.f("q_w1T"), d, d, 1);
    c.launches += enf_launch_transpose(st, w->v_w1, c.f("v_w1T"), d, d, 1);
    c.launches += enf_launch_transpose(st, c.f("Wp"), c.f("WpT"), d, d, 1);
    c.launches += enf_launch_weight_image(st, c.f("q_w1T"), c.f("img_q_w1"), nullptr, d, d, 1);
    c.launches += enf_launch_weight_image(st, c.f("v_w1T"), c.f("img_v_w1"), nullptr, d, d, 1);
    c.launches += enf_launch_weight_image(st, c.f("WpT"), c.f("img_Wp"), nullptr, d, d, 1);
    c.launches += enf_launch_weight_image_T(st, c.f("W3"), c.f("img_W3"), d, d, (int)(BZ * H));
    // ENF_FLAG_RECOMPUTE: no per-pair operand stash now; the backward rebuilds it chunk by chunk
    const bool stash = train && use_tc_bwd(D) && !(D.flags & ENF_FLAG_RECOMPUTE);
    EnfPairTcParams tp = tc_fwd_params(D, rl, *w, c, pp, train, stash);
    prof_mark(0, 0, st);
    nl = enf_launch_pairs_fwd_tc(st, d, H, tp);
    prof_mark(0, 1, st);
  } else {
    prof_mark(0, 0, st);
    nl = enf_launch_pairs_fwd_simt(st, d, pp);
    prof_mark(0, 1, st);
  }
  if (nl < 0) return fail(ENF_ERR_CUDA, "pair forward kernel could not be configured");
  c.launches += nl;

  // ---- Q: per-query tail ----------------------------------------------------------------------------
  const int out_bf16 = (D.flags & ENF_FLAG_OUT_BF16) ? 1 : 0;
  if (self) {
    // a_res = a' + (nbar P1 + b1) ; FFN(a_res) = Dense_1(LN(gelu(Dense_0(a_res)))) ; out = gelu(a' + FFN)   (nef.py:62-64, 225-226)
    c.gemm((int)BC, d, Hd, enf_mat(c.f("nbar"), Hd), enf_mat(c.f("P1"), d), enf_mat(c.f("o2p"), d), opt_bias(c.f("b1")));
    c.launches += enf_launch_add(st, c.f("o2p"), c.f("o2p"), c.f("a0"), BC * d);
    c.gemm((int)BC, d, d, enf_mat(c.f("o2p"), d), enf_mat(w->fb_w1, d), enf_mat(c.f("e1"), d), opt_bias(w->fb_b1));
    c.launches += enf_launch_ln_fwd(st, c.f("e1"), BC, d, w->fb_g, w->fb_beta, c.f("e3c"), c.f("e3"), c.f("erstd"), 1);
    c.gemm((int)BC, d, d, enf_mat(c.f("e3"), d), enf_mat(w->fb_w2, d), enf_mat(c.f("fo"), d), opt_bias(w->fb_b2));
    c.launches += enf_launch_add_gelu(st, c.f("o1p"), out, c.f("a0"), c.f("fo"), BC * d);
  } else {
  c.gemm((int)BC, Hd, Hd, enf_mat(c.f("nbar"), Hd), enf_mat(c.f("W_A"), Hd), enf_mat(c.f("e1"), Hd),
         with_lo(opt_bias(c.f("b_A")), use_tc ? c.f("lo_W_A") : nullptr));
  c.launches += enf_launch_ln_fwd(st, c.f("e1"), BC, Hd, w->fb_g, w->fb_beta, c.f("e3c"), c.f("e3"), c.f("erstd"), 1);
  if (use_tc) {
    // the tf32 kernels read their A operand with TMA, so gelu is applied by the producer (second output)
    EnfGemmOpts o;
    o.tc = 1;
    o.bias = w->fb_b2; o.gelu_out = c.f("fo_act"); o.b_lo = c.f("lo_fb_w2");
    c.gemm((int)BC, Hd, Hd, enf_mat(c.f("e3"), Hd), enf_mat(w->fb_w2, Hd), enf_mat(c.f("fo"), Hd), o);
    o.bias = w->m0_b; o.gelu_out = c.f("o1_act"); o.b_lo = c.f("lo_m0_w");
    c.gemm((int)BC, d, Hd, enf_mat(c.f("fo_act"), Hd), enf_mat(w->m0_w, d), enf_mat(c.f("o1p"), d), o);
    o.bias = w->m1_b; o.gelu_out = c.f("o2_act"); o.b_lo = c.f("lo_m1_w");
    c.gemm((int)BC, d, d, enf_mat(c.f("o1_act"), d), enf_mat(w->m1_w, d), enf_mat(c.f("o2p"), d), o);
    if (enf_thin_supported(d, O)) c.launches += enf_launch_thin_out(st, c.f("o2_act"), w->m2_w, w->m2_b, out, BC, d, O, 0, out_bf16);
    else c.gemm((int)BC, O, d, enf_mat(c.f("o2_act"), d), enf_mat(w->m2_w, O), enf_mat(out, O), opt_bias(w->m2_b));
  } else {
    c.gemm((int)BC, Hd, Hd, enf_mat(c.f("e3"), Hd), enf_mat(w->fb_w2, Hd), enf_mat(c.f("fo"), Hd), opt_bias(w->fb_b2));
    EnfGemmOpts o; o.act_a = 1;
    o.bias = w->m0_b; c.gemm((int)BC, d, Hd, enf_mat(c.f("fo"), Hd), enf_mat(w->m0_w, d), enf_mat(c.f("o1p"), d), o);
    o.bias = w->m1_b; c.gemm((int)BC, d, d, enf_mat(c.f("o1p"), d), enf_mat(w->m1_w, d), enf_mat(c.f("o2p"), d), o);
    if (enf_thin_supported(d, O)) c.launches += enf_launch_thin_out(st, c.f("o2p"), w->m2_w, w->m2_b, out, BC, d, O, 1, out_bf16);
    else { o.bias = w->m2_b; c.gemm((int)BC, O, d, enf_mat(c.f("o2p"), d), enf_mat(w->m2_w, O), enf_mat(out, O), o); }
  }
  }   // !self
  if (c.gemm_failed) return fail(ENF_ERR_CUDA, "a tensor-core stage GEMM could not be configured");
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(ENF_ERR_CUDA, std::string("CUDA error while enqueueing fwd: ") + cudaGetErrorString(e));
  {
    std::lock_guard<std::mutex> lk(g_mu);
    if (train) g_fwd_state[workspace] = FwdState{D, x_batch_stride}; else g_fwd_state.erase(workspace);
  }
  g_launches = c.launches;
  return ENF_OK;
}

}  // extern "C"
namespace {

// enf_xattn_bwd (want_dx = false: dx is not computed, whatever the flags) and enf_xattn_bwd_x
int xattn_bwd(const EnfDesc* desc, const EnfWeights* w, const float* x, int64_t x_batch_stride, const float* p,
              const float* a, const float* sigma, const float* d_out, const EnfWeightGrads* dW, float* dp, float* da,
              float* dsigma, float* dx, bool want_dx, void* workspace, size_t workspace_bytes, enf_stream_t stream) {
  g_launches = 0;
  EnfInvariantLayout rl;
  int rc = validate(desc, &rl);
  if (rc != ENF_OK) return rc;
  const EnfDesc& D = *desc;
  if (D.flags & ENF_FLAG_FORWARD_ONLY) return fail(ENF_ERR_STATE, "a forward-only description (ENF_FLAG_FORWARD_ONLY) has no backward");
  if (!d_out || !dp || !da) return fail(ENF_ERR_NULL_POINTER, "NULL argument");
  if (want_dx && dx && !(D.flags & ENF_FLAG_GRAD_X))
    return fail(ENF_ERR_STATE, "dx needs a forward run with ENF_FLAG_GRAD_X (its workspace holds the query-record cotangents)");
  if (want_dx && !dx && (D.flags & ENF_FLAG_GRAD_X)) return fail(ENF_ERR_NULL_POINTER, "dx is NULL on an ENF_FLAG_GRAD_X description");
  if (!want_dx) dx = nullptr;
  if ((rc = check_call(D, w, x, x_batch_stride, p, a, sigma, workspace)) != ENF_OK) return rc;
  {
    std::lock_guard<std::mutex> lk(g_mu);
    auto it = g_fwd_state.find(workspace);
    if (it == g_fwd_state.end() || memcmp(&it->second.D, &D, sizeof(EnfDesc)) != 0 || it->second.xbs != x_batch_stride)
      return fail(ENF_ERR_STATE, "enf_xattn_bwd needs the workspace of a matching enf_xattn_fwd call (same description, same x_batch_stride)");
  }
  Layout Y = make_layout(D, rl);
  if (workspace_bytes < Y.total * sizeof(float)) return fail(ENF_ERR_WORKSPACE, "workspace too small");

  const bool tc_fwd = tc_fwd_on(D);
  const bool tc_bwd = tc_fwd && use_tc_bwd(D);
  const bool self = (D.flags & ENF_FLAG_SELF_BLOCK) != 0, no_stem = (D.flags & ENF_FLAG_NO_STEM) != 0;
  Ctx c; c.st = (cudaStream_t)stream; c.ws = (float*)workspace; c.Y = &Y; c.tc = tc_fwd;
  cudaStream_t st = c.st;
  const int d = D.d, H = D.H, Hd = H * d, L = D.L, O = D.O;
  const int64_t BZ = (int64_t)D.B * D.Z, BC = (int64_t)D.B * D.C;
  const int Bx = (x_batch_stride == 0 && !self) ? 1 : D.B;
  auto G = [&](const char* leaf) { return c.f((std::string("gw_") + leaf).c_str()); };
  auto colsum = [&](const float* Gm, int64_t M, int N, float* out) { c.launches += enf_launch_colsum(st, Gm, M, N, N, out, nullptr, 0); };

  if (cudaMemsetAsync(c.ws + Y.acc_begin, 0, (Y.acc_end - Y.acc_begin) * sizeof(float), st) != cudaSuccess)
    return fail(ENF_ERR_CUDA, "memset of accumulators failed");

  // ---- Q backward: decode MLP, block FFN, folded (mixer Dense_1 . out_proj . FFN Dense_0) ---------------------
  // dW == NULL (latents-only backward: Meta-SGD inner loop, ODE phase): the weight-gradient products of the per-query tail
  // and of the latent stage are skipped, only the chain towards dp / da / dsigma is evaluated
  const bool wg = dW != nullptr;
  auto LO = [&](const char* name) { return tc_fwd ? c.f(name) : (const float*)nullptr; };
  if (self) {
    // backward of  out = gelu(a' + fo), fo = Dense_1(LN(gelu(Dense_0(a_res)))), a_res = a' + nbar P1 + b1
    c.launches += enf_launch_mul_gelu_grad(st, c.f("d_o1p"), d_out, c.f("o1p"), BC * d);                        // d(a' + fo)
    if (wg) {
      c.gemm(d, d, (int)BC, enf_mat(c.f("e3"), 1, d), enf_mat(c.f("d_o1p"), d), enf_mat(G("fb_w2"), d), opt_acc());
      colsum(c.f("d_o1p"), BC, d, G("fb_b2"));
    }
    c.gemm((int)BC, d, d, enf_mat(c.f("d_o1p"), d), enf_mat(w->fb_w2, 1, d), enf_mat(c.f("s1"), d));                // de3
    c.launches += enf_launch_ln_bwd(st, c.f("s1"), c.f("e3c"), c.f("erstd"), w->fb_g, c.f("e1"), BC, d, c.f("s1"),
                                    wg ? G("fb_g") : nullptr, wg ? G("fb_beta") : nullptr, 1, 0, 0);                 // de1 (in place)
    if (wg) {
      c.gemm(d, d, (int)BC, enf_mat(c.f("o2p"), 1, d), enf_mat(c.f("s1"), d), enf_mat(G("fb_w1"), d), opt_acc());
      colsum(c.f("s1"), BC, d, G("fb_b1"));
    }
    c.gemm((int)BC, d, d, enf_mat(c.f("s1"), d), enf_mat(w->fb_w1, 1, d), enf_mat(c.f("d_o2p"), d));                // d a_res
    c.launches += enf_launch_add(st, c.f("da0x"), c.f("d_o1p"), c.f("d_o2p"), BC * d);                             // both residuals -> a'
    if (wg) {
      c.gemm(Hd, d, (int)BC, enf_mat(c.f("nbar"), 1, Hd), enf_mat(c.f("d_o2p"), d), enf_mat(c.f("dP1"), d));
      if (cudaMemsetAsync(c.f("db1"), 0, d * sizeof(float), st) != cudaSuccess) return fail(ENF_ERR_CUDA, "memset failed");
      colsum(c.f("d_o2p"), BC, d, c.f("db1"));
    }
    c.gemm((int)BC, Hd, d, enf_mat(c.f("d_o2p"), d), enf_mat(c.f("P1"), 1, d), enf_mat(c.f("s0"), Hd));               // dnbar
  } else {
  {
    // wgrad A operands: gelu of the stored pre-activation (fp32 mode: applied on load; tensor-core mode: the
    // activated copies written by the forward)
    EnfGemmOpts wa = opt_acc_big(); wa.act_a = tc_fwd ? 0 : 1;
    const float* a_o2 = tc_fwd ? c.f("o2_act") : c.f("o2p");
    const float* a_o1 = tc_fwd ? c.f("o1_act") : c.f("o1p");
    const float* a_fo = tc_fwd ? c.f("fo_act") : c.f("fo");
    EnfGemmOpts o;
    o.tc = 1;
    if (enf_thin_supported(d, O)) {
      if (wg) c.launches += enf_launch_thin_wgrad(st, a_o2, d_out, G("m2_w"), G("m2_b"), BC, d, O, wa.act_a);
      c.launches += enf_launch_thin_dgrad(st, d_out, w->m2_w, c.f("o2p"), c.f("d_o2p"), BC, d, O);
    } else {
      if (wg) {
        c.gemm(d, O, (int)BC, enf_mat(a_o2, 1, d), enf_mat(d_out, O), enf_mat(G("m2_w"), O), wa);
        colsum(d_out, BC, O, G("m2_b"));
      }
      o.mul_gelu_grad = c.f("o2p");
      c.gemm((int)BC, d, O, enf_mat(d_out, O), enf_mat(w->m2_w, 1, O), enf_mat(c.f("d_o2p"), d), o);
    }
    if (wg) {
      c.gemm(d, d, (int)BC, enf_mat(a_o1, 1, d), enf_mat(c.f("d_o2p"), d), enf_mat(G("m1_w"), d), wa);
      colsum(c.f("d_o2p"), BC, d, G("m1_b"));
    }
    o.mul_gelu_grad = c.f("o1p"); o.b_lo = LO("lo_m1_w");
    c.gemm((int)BC, d, d, enf_mat(c.f("d_o2p"), d), enf_mat(w->m1_w, 1, d), enf_mat(c.f("d_o1p"), d), o);
    if (wg) {
      c.gemm(Hd, d, (int)BC, enf_mat(a_fo, 1, Hd), enf_mat(c.f("d_o1p"), d), enf_mat(G("m0_w"), d), wa);
      colsum(c.f("d_o1p"), BC, d, G("m0_b"));
    }
    o.mul_gelu_grad = c.f("fo"); o.b_lo = LO("lo_m0_w");
    c.gemm((int)BC, Hd, d, enf_mat(c.f("d_o1p"), d), enf_mat(w->m0_w, 1, d), enf_mat(c.f("s0"), Hd), o);      // dfo
  }
  if (wg) {
    c.gemm(Hd, Hd, (int)BC, enf_mat(c.f("e3"), 1, Hd), enf_mat(c.f("s0"), Hd), enf_mat(G("fb_w2"), Hd), opt_acc_big());
    colsum(c.f("s0"), BC, Hd, G("fb_b2"));
  }
  c.gemm((int)BC, Hd, Hd, enf_mat(c.f("s0"), Hd), enf_mat(w->fb_w2, 1, Hd), enf_mat(c.f("s1"), Hd),
         with_lo(EnfGemmOpts(), LO("lo_fb_w2")));                                                               // de3
  c.launches += enf_launch_ln_bwd(st, c.f("s1"), c.f("e3c"), c.f("erstd"), w->fb_g, c.f("e1"), BC, Hd, c.f("s1"),
                                  wg ? G("fb_g") : nullptr, wg ? G("fb_beta") : nullptr, 1, 0, tc_fwd ? 1 : 0);   // de1 (in place)
  if (wg) {
    c.gemm(Hd, Hd, (int)BC, enf_mat(c.f("nbar"), 1, Hd), enf_mat(c.f("s1"), Hd), enf_mat(c.f("gf_W_A"), Hd), opt_acc_big());
    colsum(c.f("s1"), BC, Hd, c.f("gf_b_A"));
  }
  c.gemm((int)BC, Hd, Hd, enf_mat(c.f("s1"), Hd), enf_mat(c.f("W_A"), 1, Hd), enf_mat(c.f("s0"), Hd),
         with_lo(EnfGemmOpts(), LO("lo_W_A")));                                                                  // dnbar
  }   // !self

  // ---- P backward --------------------------------------------------------------------------------------
  EnfPairParams pp = pair_params(D, rl, *w, c, D.use_window ? sigma : nullptr, Bx == 1 ? 0 : (int64_t)D.C * ENF_F_XI);
  int nl;
  if (tc_bwd) {
    EnfPairTcBwdParams tp;
    memset(&tp, 0, sizeof(tp));
    tp.B = D.B; tp.C = D.C; tp.Z = D.Z; tp.rec = rl;
    tp.xi = pp.xi; tp.xi_bs = pp.xi_bs; tp.lam = pp.lam; tp.sigma = pp.sigma;
    tp.q_omega = w->q_omega; tp.v_omega = w->v_omega; tp.q_b1 = w->q_b1; tp.v_b1 = w->v_b1; tp.bp = c.f("bp");
    tp.img_q_w1 = (const uint8_t*)c.f("img_q_w1"); tp.img_v_w1 = (const uint8_t*)c.f("img_v_w1");
    tp.img_Wp = (const uint8_t*)c.f("img_Wp"); tp.img_W3 = (const uint8_t*)c.f("img_W3");
    c.launches += enf_launch_weight_image(st, c.f("q_w1T"), c.f("img_q_w1_lo"), nullptr, d, d, 1, 1);
    c.launches += enf_launch_weight_image(st, c.f("v_w1T"), c.f("img_v_w1_lo"), nullptr, d, d, 1, 1);
    tp.img_q_w1_lo = (const uint8_t*)c.f("img_q_w1_lo"); tp.img_v_w1_lo = (const uint8_t*)c.f("img_v_w1_lo");
    tp.U = pp.U; tp.b3 = pp.b3; tp.slog = c.f("slog"); tp.lse = pp.lse; tp.nbar = pp.nbar;
    tp.dnbar = c.f("s0"); tp.Dg = c.f("Dg"); tp.gmax = c.f("gmax"); tp.dnb16 = reinterpret_cast<uint4*>(c.f("dnb16"));
    tp.that_img = reinterpret_cast<const uint8_t*>(c.f("that_img"));
    tp.dgr = reinterpret_cast<const uint4*>(c.f("dgr")); tp.trstd = c.f("trstd");
    tp.dthat = reinterpret_cast<__half*>(c.f("dthat")); tp.ds = c.f("ds_tc"); tp.duv = c.f("duv");
    tp.g_W3 = c.f("g_W3"); tp.g_b3 = c.f("g_b3");
    if (wg) {        // latents-only backward: kernels B / C skip the shared-weight gradient MMAs and their flush
      tp.g_q_w1 = G("q_w1"); tp.g_q_b1 = G("q_b1"); tp.g_v_w1 = G("v_w1"); tp.g_v_b1 = G("v_b1");
      tp.g_Wp = c.f("gf_Wp"); tp.g_bp = c.f("gf_bp");
    }
    tp.g_U = c.f("g_U"); tp.g_kappa = c.f("g_kappa"); tp.g_lam = c.f("g_lam"); tp.g_sigma = c.f("g_sigma");
    tp.g_xi = dx ? c.f("g_xi") : nullptr;       // kernel C's GX variant
    prof_mark(1, 0, st);
    // once per backward: the power-of-two gradient scale, the fp16 cotangent of nbar in kernel A's load order, Dg
    nl = enf_launch_pairs_bwd_tc_prep(st, d, H, tp);
    // then the three pair kernels, field chunk by field chunk.  Default: one chunk (the forward stashed the operands of
    // every field).  ENF_FLAG_RECOMPUTE: the forward kept nothing per pair; each chunk's stash is rebuilt first by re-running
    // the fused pair forward on those fields (bit-identical: same kernel, same inputs).
    const bool recompute = (D.flags & ENF_FLAG_RECOMPUTE) != 0;
    const int nb_max = chunk_fields(D);
    for (int b0 = 0; b0 < D.B && nl >= 0; b0 += nb_max) {
      const int nb = D.B - b0 < nb_max ? D.B - b0 : nb_max;
      if (recompute) {
        EnfPairTcParams fp = tc_fwd_params(D, rl, *w, c, pp, true, true);
        shift_fields(fp, D, b0, nb);
        const int r = enf_launch_pairs_fwd_tc(st, d, H, fp);
        if (r < 0) { nl = -1; break; }
        nl += r;
      }
      EnfPairTcBwdParams cp = tp;
      shift_fields(cp, D, b0, nb);
      const int r = enf_launch_pairs_bwd_tc_main(st, d, H, cp);
      if (r < 0) { nl = -1; break; }
      nl += r;
    }
    prof_mark(1, 1, st);
  } else {
    c.launches += enf_launch_transpose(st, w->q_w1, c.f("q_w1T"), d, d, 1);
    c.launches += enf_launch_transpose(st, w->v_w1, c.f("v_w1T"), d, d, 1);
    c.launches += enf_launch_transpose(st, c.f("Wp"), c.f("WpT"), d, d, 1);
    c.launches += enf_launch_transpose(st, c.f("W3"), c.f("W3T"), d, d, (int)(BZ * H));
    pp.q_w1T = c.f("q_w1T"); pp.v_w1T = c.f("v_w1T"); pp.WpT = c.f("WpT"); pp.W3T = c.f("W3T");
    pp.dnbar = c.f("s0");
    if (tc_fwd) pp.slog = c.f("slog");
    pp.g_q_w1 = G("q_w1"); pp.g_q_b1 = G("q_b1"); pp.g_v_w1 = G("v_w1"); pp.g_v_b1 = G("v_b1");
    pp.g_Wp = c.f("gf_Wp"); pp.g_bp = c.f("gf_bp");
    pp.g_W3 = c.f("g_W3"); pp.g_b3 = c.f("g_b3"); pp.g_U = c.f("g_U"); pp.g_kappa = c.f("g_kappa");
    pp.g_lam = c.f("g_lam"); pp.g_sigma = c.f("g_sigma");
    pp.g_xi = (self || dx) ? c.f("g_xi") : nullptr;
    prof_mark(1, 0, st);
    nl = enf_launch_pairs_bwd_simt(st, d, pp);
    prof_mark(1, 1, st);
  }
  if (nl < 0) return fail(ENF_ERR_CUDA, "pair backward kernel could not be configured");
  c.launches += nl;

  // ---- L backward ----------------------------------------------------------------------------------------
  if (c.gemm_failed) return fail(ENF_ERR_CUDA, "a tensor-core stage GEMM could not be configured");
  if (wg) {
    c.gemm(d, d, (int)(BZ * H * d), enf_mat(c.f("Weff"), 1, d), enf_mat(c.f("g_W3"), d), enf_mat(G("mx_w1"), d), opt_acc_big());
    c.gemm(d, d, (int)(BZ * H), enf_mat(c.f("beff"), 1, d), enf_mat(c.f("g_b3"), d), enf_mat(G("mx_w1"), d), opt_acc());
    colsum(c.f("g_b3"), BZ * H, d, G("mx_b1"));
  }
  // cotangent of Weff.  The tensor-core backward never reads the fp32 W3 (only its operand images), so it is free scratch
  // there; the fp32 backward re-reads W3 on every call and gets a buffer of its own -- either way a backward can be repeated.
  float* dWeff = tc_bwd ? c.f("W3") : c.f("dWeff");
  c.gemm((int)(BZ * H * d), d, d, enf_mat(c.f("g_W3"), d), enf_mat(w->mx_w1, 1, d), enf_mat(dWeff, d),
         with_lo(EnfGemmOpts(), LO("lo_mx_w1")));
  c.gemm((int)(BZ * H), d, d, enf_mat(c.f("g_b3"), d), enf_mat(w->mx_w1, 1, d), enf_mat(c.f("dbeff"), d));
  c.launches += enf_launch_weff_bwd(st, D, c.f("W2g"), c.f("b2g"), c.f("v0"), dWeff, c.f("dbeff"), c.f("gf_W2g"),
                                    c.f("gf_b2g"), c.f("dv0"));
  {
    EnfGemmOpts o; o.batch = H;
    // dk[bz,h,j] = sum_i A_q[i,h*d+j] dU[bz,h,i]  + dkappa[bz,h] c_q[h*d+j]
    c.gemm((int)BZ, d, d, enf_mat(c.f("g_U"), Hd, 1, d), enf_mat(c.f("A_q"), Hd, 1, d), enf_mat(c.f("dk"), Hd, 1, d), o);
    EnfGemmOpts oa = opt_acc(); oa.batch = H;
    c.gemm((int)BZ, d, 1, enf_mat(c.f("g_kappa"), H, 1, 1), enf_mat(c.f("c_q"), 0, 1, d), enf_mat(c.f("dk"), Hd, 1, d), oa);
    if (wg) {
      // dA_q[i,h*d+j] = sum_bz dU[bz,h,i] k[bz,h,j] ; dc_q[h*d+j] = sum_bz dkappa[bz,h] k[bz,h,j]
      c.gemm(d, d, (int)BZ, enf_mat(c.f("g_U"), 1, Hd, d), enf_mat(c.f("k"), Hd, 1, d), enf_mat(c.f("gf_A_q"), Hd, 1, d), oa);
      c.gemm(1, d, (int)BZ, enf_mat(c.f("g_kappa"), 0, H, 1), enf_mat(c.f("k"), Hd, 1, d), enf_mat(c.f("gf_c_q"), 0, 1, d), oa);
    }
  }
  if (wg) {
    c.gemm(d, Hd, (int)BZ, enf_mat(c.f("ahat"), 1, d), enf_mat(c.f("dk"), Hd), enf_mat(G("wk"), Hd), opt_acc());
    colsum(c.f("dk"), BZ, Hd, G("bk"));
    c.gemm(d, Hd, (int)BZ, enf_mat(c.f("ahat"), 1, d), enf_mat(c.f("dv0"), Hd), enf_mat(G("wv"), Hd), opt_acc());
    colsum(c.f("dv0"), BZ, Hd, G("bv"));
  }
  c.gemm((int)BZ, d, Hd, enf_mat(c.f("dk"), Hd), enf_mat(w->wk, 1, Hd), enf_mat(c.f("dahat"), d));
  c.gemm((int)BZ, d, Hd, enf_mat(c.f("dv0"), Hd), enf_mat(w->wv, 1, Hd), enf_mat(c.f("dahat"), d), opt_acc());
  c.launches += enf_launch_ln_bwd(st, c.f("dahat"), c.f("acore"), c.f("arstd"), w->ln_attn_g, nullptr, BZ, d, c.f("da0"),
                                  wg ? G("ln_attn_g") : nullptr, wg ? G("ln_attn_b") : nullptr, 0);
  if (self) c.launches += enf_launch_add(st, c.f("da0"), c.f("da0"), c.f("da0x"), BZ * d);      // + the two residual paths
  if (no_stem) {
    if (cudaMemcpyAsync(da, c.f("da0"), BZ * d * sizeof(float), cudaMemcpyDeviceToDevice, st) != cudaSuccess)
      return fail(ENF_ERR_CUDA, "copy of da failed");
  } else {
    if (wg) {
      c.gemm(L, d, (int)BZ, enf_mat(a, 1, L), enf_mat(c.f("da0"), d), enf_mat(G("stem_w"), d), opt_acc());
      colsum(c.f("da0"), BZ, d, G("stem_b"));
    }
    c.gemm((int)BZ, L, d, enf_mat(c.f("da0"), d), enf_mat(w->stem_w, 1, d), enf_mat(da, L));
  }
  if (self) {      // the poses in both roles: latent side through Lam, query side through xi
    c.launches += enf_launch_pose_record_bwd(st, D.invariant_kind, D.Dx, rl.P, rl.I, rl.win_kind, BZ, p, c.f("g_lam"), dp);
    c.launches += enf_launch_pose_features_bwd(st, D.invariant_kind, D.Dx, rl.P, BZ, p, c.f("g_xi"), dp);
  } else {
    c.launches += enf_launch_latent_record_bwd(st, D, p, c.f("g_lam"), dp);
    if (dx) c.launches += enf_launch_coord_features_bwd(st, D, x, Bx, c.f("g_xi"), dx);
  }
  if (dsigma) {
    if (cudaMemcpyAsync(dsigma, c.f("g_sigma"), BZ * sizeof(float), cudaMemcpyDeviceToDevice, st) != cudaSuccess)
      return fail(ENF_ERR_CUDA, "copy of dsigma failed");
  }

  // ---- W backward: unfold the folded-weight gradients --------------------------------------------------------
  if (dW) {
    // tail fold: W_A = P1 fb_w1, b_A = b1 fb_w1 + fb_b1, P1 = blockdiag(M2g) wo, b1 = tile(c2g) wo + bo
    // every product of this group reads only finished accumulators (gf_*) and weights, and writes its own leaf
    c.begin_group();
    if (!self) {
      c.gemm(Hd, Hd, Hd, enf_mat(c.f("P1"), 1, Hd), enf_mat(c.f("gf_W_A"), Hd), enf_mat(G("fb_w1"), Hd));
      c.gemm(Hd, Hd, Hd, enf_mat(c.f("gf_W_A"), Hd), enf_mat(w->fb_w1, 1, Hd), enf_mat(c.f("dP1"), Hd));
      c.gemm(1, Hd, Hd, enf_mat(c.f("gf_b_A"), Hd), enf_mat(w->fb_w1, 1, Hd), enf_mat(c.f("db1"), Hd));
    }
    c.gemm(d, d, Hd, enf_mat(c.f("gf_A_q"), Hd), enf_mat(w->wq, 1, Hd), enf_mat(G("q_wf"), d));
    c.gemm(d, Hd, d, enf_mat(w->q_wf, 1, d), enf_mat(c.f("gf_A_q"), Hd), enf_mat(G("wq"), Hd));
    c.gemm(1, d, Hd, enf_mat(c.f("gf_c_q"), Hd), enf_mat(w->wq, 1, Hd), enf_mat(G("q_bf"), d));
    c.gemm(d, d, d, enf_mat(c.f("gf_Wp"), d), enf_mat(w->fv_w1, 1, d), enf_mat(G("v_wf"), d));
    c.gemm(d, d, d, enf_mat(w->v_wf, 1, d), enf_mat(c.f("gf_Wp"), d), enf_mat(G("fv_w1"), d));
    c.gemm(1, d, d, enf_mat(c.f("gf_bp"), d), enf_mat(w->fv_w1, 1, d), enf_mat(G("v_bf"), d));
    c.gemm(1, d, 2 * Hd, enf_mat(c.f("gf_b2g"), 2 * Hd), enf_mat(w->fv_w2, 1, 2 * Hd), enf_mat(G("fv_beta"), d));
    c.end_group();
    if (self) {
      // P1_h = M2g wo_h (d, d per head), b1 = bo + sum_h c2g wo_h
      const int64_t hb = (int64_t)d * d;
      EnfGemmOpts ob; ob.batch = H;
      c.gemm(d, d, d, enf_mat(c.f("M2g"), 1, d), enf_mat(c.f("dP1"), d, 1, hb), enf_mat(G("wo"), d, 1, hb), ob);
      for (int h = 0; h < H; ++h) c.launches += enf_launch_add_outer(st, G("wo") + h * hb, d, c.f("c2g"), c.f("db1"), d, d);
      c.begin_group();
      for (int h = 0; h < H; ++h) {
        c.gemm(d, d, d, enf_mat(c.f("dP1") + h * hb, d), enf_mat(w->wo + h * hb, 1, d), enf_mat(c.f("gf_M2g"), d), opt_acc());
        c.gemm(1, d, d, enf_mat(c.f("db1"), d), enf_mat(w->wo + h * hb, 1, d), enf_mat(c.f("gf_c2g"), d), opt_acc());
      }
      c.end_group();
    } else {
    c.launches += enf_launch_add_outer(st, G("fb_w1"), Hd, c.f("b1"), c.f("gf_b_A"), Hd, Hd);
    {
      const int64_t hb = (int64_t)d * Hd;        // one head's block of rows of wo / P1
      EnfGemmOpts ob; ob.batch = H;
      c.gemm(d, Hd, d, enf_mat(c.f("M2g"), 1, d), enf_mat(c.f("dP1"), Hd, 1, hb), enf_mat(G("wo"), Hd, 1, hb), ob);
      for (int h = 0; h < H; ++h) c.launches += enf_launch_add_outer(st, G("wo") + h * hb, Hd, c.f("c2g"), c.f("db1"), d, Hd);
      c.begin_group();                 // atomic accumulations into the zero-initialised gf_M2g / gf_c2g: order-free
      for (int h = 0; h < H; ++h) {
        c.gemm(d, d, Hd, enf_mat(c.f("dP1") + h * hb, Hd), enf_mat(w->wo + h * hb, 1, Hd), enf_mat(c.f("gf_M2g"), d), opt_acc());
        c.gemm(1, d, Hd, enf_mat(c.f("db1"), Hd), enf_mat(w->wo + h * hb, 1, Hd), enf_mat(c.f("gf_c2g"), d), opt_acc());
      }
      c.end_group();
    }
    }   // !self
    c.launches += enf_launch_add_outer(st, G("wq"), Hd, w->q_bf, c.f("gf_c_q"), d, Hd);
    c.launches += enf_launch_add_outer(st, G("fv_w1"), d, w->v_bf, c.f("gf_bp"), d, d);
    c.launches += enf_launch_rowdot(st, w->fv_w2, c.f("gf_W2g"), G("fv_g"), d, 2 * Hd);
    c.launches += enf_launch_mul_rows(st, G("fv_w2"), c.f("gf_W2g"), w->fv_g, d, 2 * Hd, w->fv_beta, c.f("gf_b2g"));
    c.launches += enf_launch_rowdot(st, w->mx_w2, c.f("gf_M2g"), G("mx_g"), d, d);
    c.launches += enf_launch_mul_rows(st, G("mx_w2"), c.f("gf_M2g"), w->mx_g, d, d, w->mx_beta, c.f("gf_c2g"));
    c.gemm(1, d, d, enf_mat(c.f("gf_c2g"), d), enf_mat(w->mx_w2, 1, d), enf_mat(G("mx_beta"), d));

    // scatter the internal leaves to the caller's EnfWeightGrads (bq, fv_b1, fv_b2, mx_b2 are the folded biases' grads)
    LeafCopy t;
    size_t n[ENF_NUM_WEIGHT_LEAVES];
    leaf_sizes(D, rl.I, n);
    float* const* dst = reinterpret_cast<float* const*>(dW);
    int maxn = 0;
    for (int i = 0; i < ENF_NUM_WEIGHT_LEAVES; ++i) {
      const char* nm = kLeafNames[i];
      const float* src = G(nm);
      if (!strcmp(nm, "bq")) src = c.f("gf_c_q");
      else if (!strcmp(nm, "fv_b1")) src = c.f("gf_bp");
      else if (!strcmp(nm, "fv_b2")) src = c.f("gf_b2g");
      else if (!strcmp(nm, "mx_b2")) src = c.f("gf_c2g");
      else if (!strcmp(nm, "bo")) src = c.f("db1");
      else if (!strcmp(nm, "fb_b1") && !self) src = c.f("gf_b_A");
      t.src[i] = src; t.dst[i] = dst[i]; t.n[i] = (int)n[i];
      if ((int)n[i] > maxn) maxn = (int)n[i];
    }
    int bx = (maxn + 255) / 256; if (bx > 64) bx = 64;
    copy_leaves_kernel<<<dim3(bx, ENF_NUM_WEIGHT_LEAVES), 256, 0, st>>>(t);
    c.launches += 1;
  }
  if (c.gemm_failed) return fail(ENF_ERR_CUDA, "a tensor-core stage GEMM could not be configured");
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(ENF_ERR_CUDA, std::string("CUDA error while enqueueing bwd: ") + cudaGetErrorString(e));
  g_launches = c.launches;
  return ENF_OK;
}

}  // namespace
extern "C" {

int enf_xattn_bwd(const EnfDesc* desc, const EnfWeights* w, const float* x, int64_t x_batch_stride, const float* p,
                  const float* a, const float* sigma, const float* d_out, const EnfWeightGrads* dW, float* dp, float* da,
                  float* dsigma, void* workspace, size_t workspace_bytes, enf_stream_t stream) {
  return xattn_bwd(desc, w, x, x_batch_stride, p, a, sigma, d_out, dW, dp, da, dsigma, nullptr, false, workspace, workspace_bytes,
                   stream);
}

int enf_xattn_bwd_x(const EnfDesc* desc, const EnfWeights* w, const float* x, int64_t x_batch_stride, const float* p,
                    const float* a, const float* sigma, const float* d_out, const EnfWeightGrads* dW, float* dp, float* da,
                    float* dsigma, float* dx, void* workspace, size_t workspace_bytes, enf_stream_t stream) {
  return xattn_bwd(desc, w, x, x_batch_stride, p, a, sigma, d_out, dW, dp, da, dsigma, dx, true, workspace, workspace_bytes,
                   stream);
}

}  // extern "C"
