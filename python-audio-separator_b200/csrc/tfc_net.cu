// TFC_TDF_net forward plan (MDX23C; audio_separator/separator/uvr_lib_v5/tfc_tdf_v3.py:110-267 of the reference).
// InstanceNorm2d(affine)+GELU pre-activations, 3x3 / 1x1 / 2x2-strided convolutions, TDF linears, concat skips.
// Every contraction runs on the tcgen05 "pair" pipeline (umma_ops.cu); normalisation + GELU is one fused
// per-plane kernel between them (elementwise.cu); TDF layers too small for TMA fall back to the pair-aware SIMT GEMM.
// Activation layout: (B, C, T, F) pair tensors, F innermost (the network's own layout after transpose(-1,-2), :236).
#include <math.h>
#include <string.h>

#include <vector>

#include "common.cuh"
#include "elementwise.cuh"
#include "simt_ops.cuh"
#include "umma_ops.cuh"

namespace b200sep {

struct TNorm {
  float* gamma = nullptr;
  float* beta = nullptr;
  int c = 0;
};
struct TConv {  // any convolution routed through the umma pipeline
  void* wb_hi = nullptr;
  void* wb_lo = nullptr;
  int cin = 0, cout = 0, kc = 0, n_c = 0;
  UmmaConvPlan plan;  // bound to the tensor this layer reads
};
struct TLin {
  float* w = nullptr;    // fp32 [N][K] (SIMT fallback)
  void* w_hi = nullptr;  // bf16 [N][K]
  void* w_lo = nullptr;
  int n = 0, k = 0;
  bool umma = false;
  UmmaGemmPlan plan;
};
struct TInner {
  TNorm n1, n2, n3, n4;
  TConv tfc1, tfc2, shortcut;
  TLin lin1, lin2;
};
struct TBlock {
  std::vector<TInner> inner;
};
struct PairBuf {  // one pair tensor allocation: hi plane at p, lo plane at p + elems
  uint16_t* p = nullptr;
  int64_t elems = 0;
  void* hi() const { return p; }
  void* lo() const { return p + elems; }
};

}  // namespace b200sep

using namespace b200sep;

struct b200sep_tfcnet {
  b200sep_tfcnet_config cfg;
  int n = 0, dim_c = 0, Fs = 0;
  TConv first, final0, final2;
  std::vector<TBlock> enc, dec;
  TBlock bottleneck;
  std::vector<TNorm> down_norm, up_norm;
  std::vector<TConv> down, up;
  // activation arena, per scale i (channels c_i = c + i*g, T_i = T >> i, F_i = Fs >> i)
  std::vector<PairBuf> X, S, X1, N2, CAT, T1, NT;
  PairBuf MIX, FIRST, FC, FH;  // cws input (dim_c ch), first_conv output (c), final concat (c + dim_c), final hidden (c)
  float* out_cws = nullptr;    // fp32 (B, S*dim_c, T, Fs)
  std::vector<void*> allocs;
  int64_t device_bytes = 0;
};

namespace b200sep {

struct TReader {
  const float* p;
  int64_t n, pos = 0;
  bool ok = true;
  const float* take(int64_t c) {
    if (pos + c > n) {
      ok = false;
      return p;
    }
    const float* r = p + pos;
    pos += c;
    return r;
  }
};

static int t_alloc(b200sep_tfcnet* net, void** ptr, int64_t bytes) {
  B2_CUDA(cudaMalloc(ptr, (size_t)bytes));
  net->allocs.push_back(*ptr);
  net->device_bytes += bytes;
  return B200SEP_OK;
}
static int t_upload_f32(b200sep_tfcnet* net, float** dst, const float* src, int64_t n) {
  int rc = t_alloc(net, (void**)dst, n * 4);
  if (rc) return rc;
  B2_CUDA(cudaMemcpy(*dst, src, n * 4, cudaMemcpyHostToDevice));
  return B200SEP_OK;
}
static int t_upload_u16(b200sep_tfcnet* net, void** dst, const std::vector<uint16_t>& v) {
  int rc = t_alloc(net, dst, (int64_t)v.size() * 2);
  if (rc) return rc;
  B2_CUDA(cudaMemcpy(*dst, v.data(), v.size() * 2, cudaMemcpyHostToDevice));
  return B200SEP_OK;
}
static int t_pair(b200sep_tfcnet* net, PairBuf& b, int64_t elems) {
  b.elems = elems;
  return t_alloc(net, (void**)&b.p, elems * 4);
}

static int t_norm(b200sep_tfcnet* net, TReader& rd, TNorm& nm, int c) {
  const float* g = rd.take(c);
  const float* b = rd.take(c);
  if (!rd.ok) return B200SEP_ERR_ARG;
  nm.c = c;
  int rc = t_upload_f32(net, &nm.gamma, g, c);
  if (!rc) rc = t_upload_f32(net, &nm.beta, b, c);
  return rc;
}
enum TKind { K_CONV3, K_PW, K_DOWN, K_UP };
static int t_conv(b200sep_tfcnet* net, TReader& rd, TConv& cv, int cin, int cout, TKind kind) {
  const int taps = kind == K_CONV3 ? 9 : (kind == K_PW ? 1 : 4);
  const float* w = rd.take((int64_t)cin * cout * taps);
  if (!rd.ok) return B200SEP_ERR_ARG;
  cv.cin = cin;
  cv.cout = cout;
  std::vector<uint16_t> hi, lo;
  if (kind == K_CONV3) {
    B2_CHECK_ARG(umma_conv_supported(cin, cout, 8, 3, 3), "tfcnet: 3x3 conv %d->%d channels is not supported by the tensor-core path (need multiples of 16)", cin, cout);
    umma_conv_choose(cin, cout, &cv.kc, &cv.n_c);
    umma_conv_block_weights(w, cout, cin, cv.kc, cv.n_c, hi, lo);
  } else if (kind == K_PW) {
    B2_CHECK_ARG(umma_pw_supported(cin, cout, 8), "tfcnet: 1x1 conv %d->%d channels is not supported by the tensor-core path", cin, cout);
    umma_pw_choose(cin, cout, &cv.kc, &cv.n_c);
    umma_pw_block_weights(w, cout, cin, cv.kc, cv.n_c, hi, lo);
  } else {
    const int up = kind == K_UP;
    B2_CHECK_ARG(umma_updown_supported(cin, cout, 8, up), "tfcnet: 2x2 %s conv %d->%d channels is not supported by the tensor-core path", up ? "transposed" : "strided", cin, cout);
    umma_updown_choose(cin, cout, up, &cv.kc, &cv.n_c);
    if (up) umma_up_block_weights(w, cin, cout, cv.kc, cv.n_c, hi, lo);
    else umma_down_block_weights(w, cout, cin, cv.kc, cv.n_c, hi, lo);
  }
  int rc = t_upload_u16(net, &cv.wb_hi, hi);
  if (!rc) rc = t_upload_u16(net, &cv.wb_lo, lo);
  return rc;
}
static inline uint16_t t_f2bf(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}
static inline float t_bf2f(uint16_t h) {
  uint32_t u = (uint32_t)h << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}
static int t_lin(b200sep_tfcnet* net, TReader& rd, TLin& ln, int n, int k) {
  const float* w = rd.take((int64_t)n * k);
  if (!rd.ok) return B200SEP_ERR_ARG;
  ln.n = n;
  ln.k = k;
  int rc = t_upload_f32(net, &ln.w, w, (int64_t)n * k);
  if (!rc && umma_gemm_supported(1, n, k)) {
    std::vector<uint16_t> hi((size_t)n * k), lo(hi.size());
    for (size_t i = 0; i < hi.size(); ++i) {
      hi[i] = t_f2bf(w[i]);
      lo[i] = t_f2bf(w[i] - t_bf2f(hi[i]));
    }
    rc = t_upload_u16(net, &ln.w_hi, hi);
    if (!rc) rc = t_upload_u16(net, &ln.w_lo, lo);
    ln.umma = rc == 0;
  }
  return rc;
}
static int t_block(b200sep_tfcnet* net, TReader& rd, TBlock& blk, int in_c, int c, int f) {
  const b200sep_tfcnet_config& cfg = net->cfg;
  blk.inner.resize(cfg.l);
  for (int i = 0; i < cfg.l; ++i) {
    TInner& ib = blk.inner[i];
    int rc = t_norm(net, rd, ib.n1, in_c);
    if (!rc) rc = t_conv(net, rd, ib.tfc1, in_c, c, K_CONV3);
    if (!rc) rc = t_norm(net, rd, ib.n2, c);
    if (!rc) rc = t_lin(net, rd, ib.lin1, f / cfg.bn, f);
    if (!rc) rc = t_norm(net, rd, ib.n3, c);
    if (!rc) rc = t_lin(net, rd, ib.lin2, f, f / cfg.bn);
    if (!rc) rc = t_norm(net, rd, ib.n4, c);
    if (!rc) rc = t_conv(net, rd, ib.tfc2, c, c, K_CONV3);
    if (!rc) rc = t_conv(net, rd, ib.shortcut, in_c, c, K_PW);
    if (rc) return rc;
    in_c = c;
  }
  return B200SEP_OK;
}
static int64_t t_block_params(const b200sep_tfcnet_config& c, int64_t in_c, int64_t ch, int64_t f) {
  int64_t t = 0;
  for (int i = 0; i < c.l; ++i) {
    t += 2 * in_c + ch * in_c * 9 + 2 * ch + (f / c.bn) * f + 2 * ch + f * (f / c.bn) + 2 * ch + ch * ch * 9 + ch * in_c;
    in_c = ch;
  }
  return t;
}

// bind a conv layer's TMA plan to its input tensor (B, cin, T, F)
static int t_bind(const b200sep_tfcnet* net, TConv& cv, const PairBuf& in, int T, int F) {
  return umma_conv_plan_create(&cv.plan, in.hi(), in.lo(), net->cfg.max_batch, cv.cin, T, F, cv.kc);
}
static int t_bind_lin(const b200sep_tfcnet* net, TLin& ln, const PairBuf& a, int M) {
  if (!ln.umma) return B200SEP_OK;
  return umma_gemm_plan_create(&ln.plan, a.hi(), a.lo(), ln.w_hi, ln.w_lo, M, ln.n, ln.k);
}
static int t_bind_block(b200sep_tfcnet* net, TBlock& blk, int scale, const PairBuf& xin, int c, int T, int F) {
  const PairBuf* in = &xin;
  const int M = net->cfg.max_batch * c * T;
  for (size_t i = 0; i < blk.inner.size(); ++i) {
    TInner& ib = blk.inner[i];
    int rc = t_bind(net, ib.shortcut, *in, T, F);
    if (!rc) rc = t_bind(net, ib.tfc1, net->N2[scale], T, F);
    if (!rc) rc = t_bind_lin(net, ib.lin1, net->N2[scale], M);
    if (!rc) rc = t_bind_lin(net, ib.lin2, net->NT[scale], M);
    if (!rc) rc = t_bind(net, ib.tfc2, net->N2[scale], T, F);
    if (rc) return rc;
    in = &net->X[scale];
  }
  return B200SEP_OK;
}

static int t_linear(const TLin& ln, const PairBuf& a, int M, const PairBuf& out, const PairBuf* res, cudaStream_t st) {
  if (ln.umma) {
    UmmaEpilogue e;
    e.out_hi = out.hi(); e.out_lo = out.lo();
    if (res) { e.res_hi = res->hi(); e.res_lo = res->lo(); }
    return umma_gemm_run_ex(ln.plan, 1, 1, M, e, st);
  }
  GemmParams g;
  g.A = (const float*)a.hi(); g.A_lo = a.lo(); g.Bw = ln.w; g.scale = nullptr; g.shift = nullptr;
  g.res = res ? (const float*)res->hi() : nullptr; g.res_lo = res ? res->lo() : nullptr;
  g.C = (float*)out.hi(); g.C_lo = out.lo();
  g.M = M; g.N = ln.n; g.K = ln.k; g.rows_per_channel = 1; g.channels = 1; g.relu = 0;
  return gemm_tn_simt(g, st);
}

// One TFC_TDF stack (tfc_tdf_v3.py:140-148).  xin: (B, in_c, T, F); result -> `out` (channels [out_off, out_off+c) of out_total),
// optionally multiplied by `mul` (the `x * first_conv_out` of :255 folded into the last block).
static int t_run_block(b200sep_tfcnet* net, TBlock& blk, int scale, const PairBuf& xin, int in_c, int c, int T, int F, const PairBuf& out, int out_total, int out_off,
                       const PairBuf* mul, int B, cudaStream_t st) {
  const PairBuf* in = &xin;
  const int64_t P = (int64_t)T * F;
  const int M = B * c * T;
  const int bn = net->cfg.bn;
  int rc;
  for (size_t i = 0; i < blk.inner.size(); ++i) {
    TInner& ib = blk.inner[i];
    const bool last = i + 1 == blk.inner.size();
    UmmaEpilogue e;
    // s = shortcut(x)
    e.out_hi = net->S[scale].hi(); e.out_lo = net->S[scale].lo();
    rc = umma_pw_run_ex(ib.shortcut.plan, ib.shortcut.wb_hi, ib.shortcut.wb_lo, B, c, ib.shortcut.n_c, e, st);
    if (rc) return rc;
    // x1 = tfc1(act(norm(x)))
    rc = instnorm_act_pair(in->hi(), in->lo(), in_c, 0, ib.n1.gamma, ib.n1.beta, 2, net->N2[scale].hi(), net->N2[scale].lo(), B, in_c, P, st);
    if (rc) return rc;
    e = UmmaEpilogue();
    e.out_hi = net->X1[scale].hi(); e.out_lo = net->X1[scale].lo();
    rc = umma_conv_run_ex(ib.tfc1.plan, ib.tfc1.wb_hi, ib.tfc1.wb_lo, B, c, ib.tfc1.n_c, e, st);
    if (rc) return rc;
    // x1 += tdf(x1): lin2(act(norm(lin1(act(norm(x1))))))
    rc = instnorm_act_pair(net->X1[scale].hi(), net->X1[scale].lo(), c, 0, ib.n2.gamma, ib.n2.beta, 2, net->N2[scale].hi(), net->N2[scale].lo(), B, c, P, st);
    if (rc) return rc;
    rc = t_linear(ib.lin1, net->N2[scale], M, net->T1[scale], nullptr, st);
    if (rc) return rc;
    rc = instnorm_act_pair(net->T1[scale].hi(), net->T1[scale].lo(), c, 0, ib.n3.gamma, ib.n3.beta, 2, net->NT[scale].hi(), net->NT[scale].lo(), B, c, (int64_t)T * (F / bn), st);
    if (rc) return rc;
    rc = t_linear(ib.lin2, net->NT[scale], M, net->X1[scale], &net->X1[scale], st);  // in-place residual
    if (rc) return rc;
    // x = tfc2(act(norm(x1))) + s
    rc = instnorm_act_pair(net->X1[scale].hi(), net->X1[scale].lo(), c, 0, ib.n4.gamma, ib.n4.beta, 2, net->N2[scale].hi(), net->N2[scale].lo(), B, c, P, st);
    if (rc) return rc;
    e = UmmaEpilogue();
    e.res_hi = net->S[scale].hi(); e.res_lo = net->S[scale].lo();
    if (last) {
      e.out_hi = out.hi(); e.out_lo = out.lo(); e.out_c_total = out_total; e.out_c_off = out_off;
      if (mul) { e.mul_hi = mul->hi(); e.mul_lo = mul->lo(); }
    } else {
      e.out_hi = net->X[scale].hi(); e.out_lo = net->X[scale].lo();
    }
    rc = umma_conv_run_ex(ib.tfc2.plan, ib.tfc2.wb_hi, ib.tfc2.wb_lo, B, c, ib.tfc2.n_c, e, st);
    if (rc) return rc;
    in = &net->X[scale];
    in_c = c;
  }
  return B200SEP_OK;
}

}  // namespace b200sep

extern "C" int64_t b200sep_tfcnet_param_count(const b200sep_tfcnet_config* c) {
  if (!c || c->num_scales < 1 || c->bn < 1 || c->num_subbands < 1) return -1;
  const int64_t dim_c = (int64_t)c->num_subbands * c->audio_channels * 2;
  int64_t f = c->dim_f / c->num_subbands, ch = c->c, total = ch * dim_c;
  for (int i = 0; i < c->num_scales; ++i) {
    total += t_block_params(*c, ch, ch, f) + 2 * ch + (ch + c->g) * ch * 4;
    f /= 2;
    ch += c->g;
  }
  total += t_block_params(*c, ch, ch, f);
  for (int i = 0; i < c->num_scales; ++i) {
    total += 2 * ch + ch * (ch - c->g) * 4;
    f *= 2;
    ch -= c->g;
    total += t_block_params(*c, 2 * ch, ch, f);
  }
  total += ch * (ch + dim_c) + (int64_t)c->num_targets * dim_c * ch;
  return total;
}

extern "C" void b200sep_tfcnet_destroy(b200sep_tfcnet* net) {
  if (!net) return;
  for (void* p : net->allocs) cudaFree(p);
  delete net;
}

extern "C" int b200sep_tfcnet_create(b200sep_tfcnet** out, const b200sep_tfcnet_config* cfg, const float* params_host, int64_t n_params) {
  B2_CHECK_ARG(out && cfg && params_host, "tfcnet_create: NULL argument");
  B2_CHECK_ARG(cfg->audio_channels == 2, "tfcnet_create: stereo only");
  B2_CHECK_ARG(cfg->num_scales >= 1 && cfg->l >= 1 && cfg->max_batch >= 1 && cfg->num_targets >= 1, "tfcnet_create: bad config");
  const int n = cfg->num_scales;
  const int Fs = cfg->dim_f / cfg->num_subbands;
  B2_CHECK_ARG(cfg->dim_f % cfg->num_subbands == 0 && Fs % (1 << n) == 0 && cfg->dim_t % (1 << n) == 0, "tfcnet_create: dim_f/num_subbands=%d and dim_t=%d must be divisible by 2^%d", Fs,
               cfg->dim_t, n);
  B2_CHECK_ARG(((Fs >> n) % cfg->bn) == 0 && (Fs >> n) % 8 == 0, "tfcnet_create: innermost frequency size %d must be a multiple of 8 and of bn", Fs >> n);
  // the instance norm of the TDF hidden layer works on planes of (T >> i) * ((Fs >> i) / bn) elements in groups of 8; the bottleneck's is the smallest
  // (every larger scale's is 4x the next one's)
  B2_CHECK_ARG((int64_t)(cfg->dim_t >> n) * ((Fs >> n) / cfg->bn) % 8 == 0,
               "tfcnet_create: the bottleneck's TDF hidden plane (dim_t>>%d) * ((dim_f/num_subbands>>%d)/bn) = %d * %d must be a multiple of 8", n, n, cfg->dim_t >> n,
               (Fs >> n) / cfg->bn);
  const int64_t expect = b200sep_tfcnet_param_count(cfg);
  B2_CHECK_ARG(expect == n_params, "tfcnet_create: expected %lld parameters for this config, got %lld", (long long)expect, (long long)n_params);
  int devs = 0;
  B2_CUDA(cudaGetDeviceCount(&devs));

  b200sep_tfcnet* net = new b200sep_tfcnet();
  net->cfg = *cfg;
  net->n = n;
  net->dim_c = cfg->num_subbands * cfg->audio_channels * 2;
  net->Fs = Fs;
  const int dim_c = net->dim_c, c0 = cfg->c, g = cfg->g, T0 = cfg->dim_t, Bm = cfg->max_batch;
  TReader rd{params_host, n_params};
  int rc = t_conv(net, rd, net->first, dim_c, c0, K_PW);
  net->enc.resize(n); net->dec.resize(n); net->down.resize(n); net->up.resize(n); net->down_norm.resize(n); net->up_norm.resize(n);
  int f = Fs, c = c0;
  for (int i = 0; i < n && !rc; ++i) {
    rc = t_block(net, rd, net->enc[i], c, c, f);
    if (!rc) rc = t_norm(net, rd, net->down_norm[i], c);
    if (!rc) rc = t_conv(net, rd, net->down[i], c, c + g, K_DOWN);
    f /= 2; c += g;
  }
  if (!rc) rc = t_block(net, rd, net->bottleneck, c, c, f);
  for (int i = 0; i < n && !rc; ++i) {
    rc = t_norm(net, rd, net->up_norm[i], c);
    if (!rc) rc = t_conv(net, rd, net->up[i], c, c - g, K_UP);
    f *= 2; c -= g;
    if (!rc) rc = t_block(net, rd, net->dec[i], 2 * c, c, f);
  }
  if (!rc) rc = t_conv(net, rd, net->final0, c + dim_c, c, K_PW);
  if (!rc) rc = t_conv(net, rd, net->final2, c, cfg->num_targets * dim_c, K_PW);
  if (!rc && (!rd.ok || rd.pos != n_params)) {
    set_error("tfcnet_create: parameter blob size mismatch (consumed %lld of %lld)", (long long)rd.pos, (long long)n_params);
    rc = B200SEP_ERR_ARG;
  }
  // ---- activation arena
  net->X.resize(n + 1); net->S.resize(n + 1); net->X1.resize(n + 1); net->N2.resize(n + 1); net->CAT.resize(n + 1); net->T1.resize(n + 1); net->NT.resize(n + 1);
  for (int i = 0; i <= n && !rc; ++i) {
    const int64_t ci = c0 + (int64_t)i * g, Ti = T0 >> i, Fi = Fs >> i;
    const int64_t e = (int64_t)Bm * ci * Ti * Fi;
    rc = t_pair(net, net->X[i], e);
    if (!rc) rc = t_pair(net, net->S[i], e);
    if (!rc) rc = t_pair(net, net->X1[i], e);
    if (!rc) rc = t_pair(net, net->N2[i], i < n ? 2 * e : e);
    if (!rc && i < n) rc = t_pair(net, net->CAT[i], 2 * e);
    if (!rc) rc = t_pair(net, net->T1[i], (int64_t)Bm * ci * Ti * (Fi / cfg->bn));
    if (!rc) rc = t_pair(net, net->NT[i], (int64_t)Bm * ci * Ti * (Fi / cfg->bn));
  }
  const int64_t px = (int64_t)Bm * T0 * Fs;
  if (!rc) rc = t_pair(net, net->MIX, px * dim_c);
  if (!rc) rc = t_pair(net, net->FIRST, px * c0);
  if (!rc) rc = t_pair(net, net->FC, px * (c0 + dim_c));
  if (!rc) rc = t_pair(net, net->FH, px * c0);
  if (!rc) rc = t_alloc(net, (void**)&net->out_cws, px * cfg->num_targets * dim_c * 4);
  // ---- bind TMA plans to the buffers each layer reads
  if (!rc) rc = t_bind(net, net->first, net->MIX, T0, Fs);
  for (int i = 0; i < n && !rc; ++i) {
    const int ci = c0 + i * g, Ti = T0 >> i, Fi = Fs >> i;
    rc = t_bind_block(net, net->enc[i], i, i == 0 ? net->FIRST : net->X[i], ci, Ti, Fi);
    if (!rc) rc = t_bind(net, net->down[i], net->N2[i], Ti, Fi);
  }
  if (!rc) rc = t_bind_block(net, net->bottleneck, n, net->X[n], c0 + n * g, T0 >> n, Fs >> n);
  for (int i = 0; i < n && !rc; ++i) {
    const int s = n - 1 - i;  // decoder block i works at scale s
    const int cs = c0 + s * g, Ts = T0 >> s, Fsz = Fs >> s;
    rc = t_bind(net, net->up[i], net->N2[s + 1], Ts / 2, Fsz / 2);
    if (!rc) rc = t_bind_block(net, net->dec[i], s, net->CAT[s], cs, Ts, Fsz);
  }
  if (!rc) rc = t_bind(net, net->final0, net->FC, T0, Fs);
  if (!rc) rc = t_bind(net, net->final2, net->FH, T0, Fs);
  if (rc) {
    b200sep_tfcnet_destroy(net);
    return rc;
  }
  *out = net;
  return B200SEP_OK;
}

extern "C" int64_t b200sep_tfcnet_device_bytes(const b200sep_tfcnet* net) { return net ? net->device_bytes : 0; }

extern "C" int b200sep_tfcnet_forward(b200sep_tfcnet* net, const float* spec_in, float* spec_out, int batch, void* stream) {
  B2_CHECK_ARG(net && spec_in && spec_out, "tfcnet_forward: NULL argument");
  B2_CHECK_ARG(batch >= 0 && batch <= net->cfg.max_batch, "tfcnet_forward: batch=%d exceeds max_batch=%d", batch, net->cfg.max_batch);
  if (batch == 0) return B200SEP_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const b200sep_tfcnet_config& cfg = net->cfg;
  const int n = net->n, B = batch, dim_c = net->dim_c, K = cfg.num_subbands, Fs = net->Fs, T0 = cfg.dim_t, c0 = cfg.c, g = cfg.g;
  // cac2cws (:216-221) into the first conv's input and into channels [0, dim_c) of the final concat (torch.cat([mix, x]), :257)
  int rc = cws_split_pair(spec_in, net->MIX.hi(), net->MIX.lo(), B, 4, T0, K, Fs, dim_c, 0, st);
  if (!rc) rc = cws_split_pair(spec_in, net->FC.hi(), net->FC.lo(), B, 4, T0, K, Fs, c0 + dim_c, 0, st);
  if (rc) return rc;
  UmmaEpilogue e;
  e.out_hi = net->FIRST.hi(); e.out_lo = net->FIRST.lo();
  rc = umma_pw_run_ex(net->first.plan, net->first.wb_hi, net->first.wb_lo, B, c0, net->first.n_c, e, st);  // first_conv (:234)
  if (rc) return rc;
  int c = c0, T = T0, F = Fs;
  for (int i = 0; i < n; ++i) {  // encoder (:239-242): block output goes straight into the second half of the decoder's concat buffer
    rc = t_run_block(net, net->enc[i], i, i == 0 ? net->FIRST : net->X[i], c, c, T, F, net->CAT[i], 2 * c, c, nullptr, B, st);
    if (rc) return rc;
    rc = instnorm_act_pair(net->CAT[i].hi(), net->CAT[i].lo(), 2 * c, c, net->down_norm[i].gamma, net->down_norm[i].beta, 2, net->N2[i].hi(), net->N2[i].lo(), B, c, (int64_t)T * F, st);
    if (rc) return rc;
    e = UmmaEpilogue();
    e.out_hi = net->X[i + 1].hi(); e.out_lo = net->X[i + 1].lo();
    rc = umma_down_run_ex(net->down[i].plan, net->down[i].wb_hi, net->down[i].wb_lo, B, c + g, net->down[i].n_c, e, st);
    if (rc) return rc;
    c += g; T /= 2; F /= 2;
  }
  rc = t_run_block(net, net->bottleneck, n, net->X[n], c, c, T, F, net->X[n], c, 0, nullptr, B, st);  // :244
  if (rc) return rc;
  for (int i = 0; i < n; ++i) {  // decoder (:246-249)
    const int s = n - 1 - i;
    rc = instnorm_act_pair(net->X[s + 1].hi(), net->X[s + 1].lo(), c, 0, net->up_norm[i].gamma, net->up_norm[i].beta, 2, net->N2[s + 1].hi(), net->N2[s + 1].lo(), B, c, (int64_t)T * F, st);
    if (rc) return rc;
    e = UmmaEpilogue();
    e.out_hi = net->CAT[s].hi(); e.out_lo = net->CAT[s].lo(); e.out_c_total = 2 * (c - g); e.out_c_off = 0;
    rc = umma_up_run_ex(net->up[i].plan, net->up[i].wb_hi, net->up[i].wb_lo, B, c - g, net->up[i].n_c, e, st);
    if (rc) return rc;
    c -= g; T *= 2; F *= 2;
    const bool last = s == 0;  // the last decoder block writes x * first_conv_out into channels [dim_c, dim_c + c) of the final concat
    rc = t_run_block(net, net->dec[i], s, net->CAT[s], 2 * c, c, T, F, last ? net->FC : net->X[s], last ? c0 + dim_c : c, last ? dim_c : 0, last ? &net->FIRST : nullptr, B, st);
    if (rc) return rc;
  }
  e = UmmaEpilogue();  // final_conv: 1x1 -> GELU -> 1x1 (:257)
  e.out_hi = net->FH.hi(); e.out_lo = net->FH.lo(); e.act = 2;
  rc = umma_pw_run_ex(net->final0.plan, net->final0.wb_hi, net->final0.wb_lo, B, c0, net->final0.n_c, e, st);
  if (rc) return rc;
  e = UmmaEpilogue();
  e.out_f32 = net->out_cws;
  rc = umma_pw_run_ex(net->final2.plan, net->final2.wb_hi, net->final2.wb_lo, B, cfg.num_targets * dim_c, net->final2.n_c, e, st);
  if (rc) return rc;
  return cws_merge_f32(net->out_cws, spec_out, B, cfg.num_targets, 4, T0, K, Fs, st);  // cws2cac + (B,S,4,F,T) view (:259-263)
}
