// Native layer runtime: launches the whole per-layer kernel sequence of a BertLayer stack
// (forward and backward) from C++, so the host cost per step is a handful of calls instead of
// hundreds of Python->ctypes round trips. Pure orchestration: every arithmetic step is one of the
// kernels behind the C-ABI (gemm_tcgen05, attention_tc, rowwise).
#include <stdlib.h>
#include <string.h>

#include "common.h"

namespace hero {

enum { ACT_NONE = 0, ACT_GELU = 1, ACT_RELU = 2, ACT_GELU_GRAD = 3 };

static inline uint32_t site_key(uint32_t base, int layer, int site) {
  uint32_t h = base ^ (0x9E3779B1u * (uint32_t)(layer * 4 + site + 1));
  h ^= h >> 16; h *= 0x85EBCA6Bu; h ^= h >> 13; h *= 0xC2B2AE35u; h ^= h >> 16;
  return h;
}

struct Gemm {
  hero_gemm_args g;
  Gemm(const void* a, long long lda, int a_mn, const void* b, long long ldb, int b_mn, int m, int n,
       int k, void* out, long long ld_out) {
    memset(&g, 0, sizeof(g));
    g.a = a; g.lda = lda; g.a_mn_major = a_mn;
    g.b = b; g.ldb = ldb; g.b_mn_major = b_mn;
    g.m = m; g.n = n; g.k = k;
    g.out = out; g.ld_out = ld_out;
    g.drop_scale = 1.0f;
  }
  Gemm& bias(const float* p) { g.bias = p; return *this; }
  Gemm& resid(const void* p, long long ld) { g.resid = p; g.ld_resid = ld; return *this; }
  // fp32 residual in, fp32 pre-LayerNorm sum out (the residual stream of the forward pass)
  Gemm& resid_f32(const float* p, long long ld) {
    g.resid = p; g.ld_resid = ld; g.resid_f32 = 1; g.out_f32_store = 1; return *this;
  }
  // ... with the residual given as a pre-LayerNorm sum + its statistics and affine parameters
  Gemm& resid_ln(const float* sum, long long ld, const float* mean, const float* rstd,
                 const float* gamma, const float* beta) {
    resid_f32(sum, ld);
    g.resid_ln_mean = mean; g.resid_ln_rstd = rstd; g.resid_ln_gamma = gamma; g.resid_ln_beta = beta;
    return *this;
  }
  Gemm& act(int a) { g.act = a; return *this; }
  Gemm& aux_out(void* p, long long ld) { g.aux_out = p; g.ld_aux_out = ld; return *this; }
  Gemm& aux_in(const void* p, long long ld) { g.aux_in = p; g.ld_aux_in = ld; return *this; }
  Gemm& drop(uint32_t thr, uint32_t key, float scale) {
    g.drop_threshold = thr; g.drop_key = key; g.drop_scale = scale; return *this;
  }
  Gemm& f32_accumulate() { g.out_f32_accumulate = 1; return *this; }
  // column sums of the stored output accumulate into p (bias gradient of the producing Linear)
  Gemm& colsum(float* p) { g.out_colsum = p; return *this; }
  int run(void* stream) { return hero_gemm_bf16(&g, stream); }
};

static void ln_base(hero_ln_args* a, const void* x, const float* gamma, const float* beta, float eps,
                    int n_rows, int h, float* mean, float* rstd) {
  memset(a, 0, sizeof(*a));
  a->x = x; a->x_is_f32 = 1; a->gamma = gamma; a->beta = beta; a->eps = eps;
  a->n_rows = n_rows; a->h = h; a->mean = mean; a->rstd = rstd;
  a->x_pad_idx = -1; a->add_pad_idx = -1;
  a->drop_scale = 1.0f; a->drop2_scale = 1.0f;
}

// Weight-gradient stream. The backward of a layer is a dependency chain (LN' -> dgrad GEMMs ->
// attention') plus four weight-gradient GEMMs and two bias column sums that hang off it and are
// consumed only by the optimizer. They run on a library-owned second stream, ordered by events,
// so their CTAs fill the SMs that the chain's kernels leave idle: launch gaps, wave tails, and
// half of the machine for the 25-block GEMMs of the 3200-token temporal encoder.
struct SideStream {
  int device = -1;
  cudaStream_t stream = nullptr;
  cudaEvent_t ready = nullptr;     // chain -> side: an operand of the next weight gradient exists
  cudaEvent_t done[2] = {nullptr, nullptr};   // side -> chain: layer's reads of scratch[parity] over
  cudaEvent_t joined = nullptr;
};

static int side_stream(SideStream** out) {
  static SideStream ctx[16];
  int dev = 0;
  HERO_CUDA_CHECK(cudaGetDevice(&dev));
  HERO_REQUIRE(dev >= 0 && dev < 16, "stack: unsupported device ordinal %d", dev);
  SideStream& c = ctx[dev];
  if (c.stream == nullptr) {
    HERO_CUDA_CHECK(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
    HERO_CUDA_CHECK(cudaEventCreateWithFlags(&c.ready, cudaEventDisableTiming));
    HERO_CUDA_CHECK(cudaEventCreateWithFlags(&c.done[0], cudaEventDisableTiming));
    HERO_CUDA_CHECK(cudaEventCreateWithFlags(&c.done[1], cudaEventDisableTiming));
    HERO_CUDA_CHECK(cudaEventCreateWithFlags(&c.joined, cudaEventDisableTiming));
    c.device = dev;
  }
  *out = &c;
  return HERO_OK;
}

#define HERO_TRY(expr)        \
  do {                        \
    int _rc = (expr);         \
    if (_rc) return _rc;      \
  } while (0)

// Timing ablations (tools/ablate.sh builds a second library with -DHERO_ABLATE; never defined in
// the product build): HERO_ABLATE=<bit mask> skips whole kernel families inside the stack so a
// bench run shows what each family really costs in the overlapped step. Results are garbage.
#ifdef HERO_ABLATE
static int ablate(int bit) {
  static int mask = -1;
  if (mask < 0) {
    const char* e = getenv("HERO_ABLATE");
    mask = e ? atoi(e) : 0;
  }
  return (mask >> bit) & 1;
}
#define HERO_STEP(bit, expr) do { if (!ablate(bit)) HERO_TRY(expr); } while (0)
#else
#define HERO_STEP(bit, expr) HERO_TRY(expr)
#endif
enum { ABL_COLSUM = 0, ABL_ATTN_FWD, ABL_ATTN_BWD, ABL_LN_FWD, ABL_LN_BWD, ABL_WGRAD, ABL_DGRAD,
       ABL_FWD_GEMM };

static int check_stack(const hero_stack_args* s, bool bwd) {
  HERO_REQUIRE(s != nullptr, "null stack args");
  HERO_REQUIRE(s->n_layers >= 0 && s->n_tok > 0 && s->hidden > 0 && s->inter > 0 && s->heads > 0,
               "bad stack dims");
  HERO_REQUIRE(s->hidden == s->heads * 64, "stack: hidden must be heads * 64");
  HERO_REQUIRE(s->weights && s->acts && s->x, "stack: null weights/acts/x");
  HERO_REQUIRE(s->tile_tok0 && s->tile_ntok && s->seq_lo && s->seq_hi, "stack: null attention plan");
  if (bwd) HERO_REQUIRE(s->grads && s->dout && s->scratch, "stack bwd: null grads/dout/scratch");
  if (!bwd) HERO_REQUIRE(s->x_f32 != nullptr, "stack fwd: null x_f32 (fp32 copy of the input)");
  return HERO_OK;
}

}  // namespace hero

using namespace hero;

extern "C" int64_t hero_bert_stack_bwd_scratch_bytes(int32_t n_tok, int32_t hidden, int32_t inter) {
  // per layer parity (x2: the weight-gradient stream may still read layer l's while layer l-1 is
  // being written): ds2, ds2_d, ds1, ds1_d [n_tok, H], dpre [n_tok, I], dqkv [n_tok, 3H];
  // single: da, dcx, dx_a, dx_b [n_tok, H]
  const int64_t row = 2 * ((int64_t)(4 + 3) * hidden + inter) + 4 * (int64_t)hidden;
  return ((int64_t)n_tok * row * 2 + 1023) / 1024 * 1024 + 1024 * 16;
}

extern "C" int hero_bert_stack_fwd(const hero_stack_args* s, void* stream) {
  HERO_TRY(check_stack(s, false));
  const int M = s->n_tok, H = s->hidden, I = s->inter;
  const float scale = 0.125f;
  const void* h = s->x;          // bf16: GEMM operand
  for (int l = 0; l < s->n_layers; ++l) {
    const hero_layer_weights& W = s->weights[l];
    const hero_layer_acts& A = s->acts[l];
    HERO_REQUIRE(A.s1 && A.s2, "stack fwd: layer %d misses its fp32 pre-LayerNorm buffers", l);
    HERO_STEP(ABL_FWD_GEMM, Gemm(h, H, 0, W.wqkv, H, 0, M, 3 * H, H, A.qkv, 3 * H).bias(W.bqkv).run(stream));
    HERO_STEP(ABL_ATTN_FWD, hero_attn_fwd(A.qkv, s->tile_tok0, s->tile_ntok, s->seq_lo, s->seq_hi, A.cx, A.lse, M,
                           s->n_tiles, s->n_long, s->max_long, s->heads, 64, scale,
                           s->attn_drop_threshold,
                           site_key(s->drop_key, l, 0), s->attn_drop_scale, stream));
    // residual of the attention block = this layer's input in fp32: the caller's fp32 copy for
    // layer 0, LayerNorm(previous layer's s2) recomputed in the epilogue afterwards
    Gemm outp(A.cx, H, 0, W.wo, H, 0, M, H, H, A.s1, H);
    outp.bias(W.bo).drop(s->hidden_drop_threshold, site_key(s->drop_key, l, 1),
                         s->hidden_drop_scale);
    if (l == 0) {
      outp.resid_f32(s->x_f32, H);
    } else {
      const hero_layer_acts& P = s->acts[l - 1];
      const hero_layer_weights& PW = s->weights[l - 1];
      outp.resid_ln(P.s2, H, P.mean2, P.rstd2, PW.ln2_g, PW.ln2_b);
    }
    HERO_STEP(ABL_FWD_GEMM, outp.run(stream));
    hero_ln_args ln;
    ln_base(&ln, A.s1, W.ln1_g, W.ln1_b, s->eps, M, H, A.mean1, A.rstd1);
    ln.y = A.a;
    HERO_STEP(ABL_LN_FWD, hero_ln_fwd(&ln, stream));
    Gemm up(A.a, H, 0, W.w1, H, 0, M, I, H, A.f, I);
    up.bias(W.b1).act(ACT_GELU);
    if (A.pre) up.aux_out(A.pre, I);
    HERO_STEP(ABL_FWD_GEMM, up.run(stream));
    HERO_STEP(ABL_FWD_GEMM, Gemm(A.f, I, 0, W.w2, I, 0, M, H, I, A.s2, H)
                 .bias(W.b2)
                 .resid_ln(A.s1, H, A.mean1, A.rstd1, W.ln1_g, W.ln1_b)
                 .drop(s->hidden_drop_threshold, site_key(s->drop_key, l, 2), s->hidden_drop_scale)
                 .run(stream));
    ln_base(&ln, A.s2, W.ln2_g, W.ln2_b, s->eps, M, H, A.mean2, A.rstd2);
    ln.y = A.out;
    ln.y_f32 = A.out_f32;      // NULL except where the caller wants the fp32 result (last layer)
    HERO_STEP(ABL_LN_FWD, hero_ln_fwd(&ln, stream));
    h = A.out;
  }
  return HERO_OK;
}

extern "C" int hero_bert_stack_bwd(const hero_stack_args* s, void* stream) {
  HERO_TRY(check_stack(s, true));
  const int M = s->n_tok, H = s->hidden, I = s->inter;
  const float scale = 0.125f;
  // carve the scratch buffer (bf16 elements)
  char* p = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(s->scratch) + 1023) &
                                    ~static_cast<uintptr_t>(1023));
  auto take = [&](long long elems) {
    char* r = p;
    p += (elems * 2 + 1023) / 1024 * 1024;
    return reinterpret_cast<void*>(r);
  };
  void *ds2_[2], *ds2_d_[2], *ds1_[2], *ds1_d_[2], *dpre_[2], *dqkv_[2];
  for (int p2 = 0; p2 < 2; ++p2) {
    ds2_[p2] = take((long long)M * H);
    ds2_d_[p2] = take((long long)M * H);
    ds1_[p2] = take((long long)M * H);
    ds1_d_[p2] = take((long long)M * H);
    dpre_[p2] = take((long long)M * I);
    dqkv_[p2] = take((long long)M * 3 * H);
  }
  void* da = take((long long)M * H);
  void* dcx = take((long long)M * H);
  void* dxa = take((long long)M * H);
  void* dxb = take((long long)M * H);

  // weight gradients on the second stream unless per-launch GEMM timing is on
  cudaStream_t chain = reinterpret_cast<cudaStream_t>(stream);
  SideStream* side = nullptr;
  const bool two_streams = !gemm_profile_active() && !serial_profiling();
  if (two_streams) HERO_TRY(side_stream(&side));
  void* wstream = two_streams ? reinterpret_cast<void*>(side->stream) : stream;
  // an operand of the next weight gradient has just been produced on the chain
  auto publish = [&]() -> int {
    if (!two_streams) return HERO_OK;
    HERO_CUDA_CHECK(cudaEventRecord(side->ready, chain));
    HERO_CUDA_CHECK(cudaStreamWaitEvent(side->stream, side->ready, 0));
    return HERO_OK;
  };
  bool done_recorded[2] = {false, false};

  const void* dy = s->dout;
  for (int l = s->n_layers - 1; l >= 0; --l) {
    const hero_layer_weights& W = s->weights[l];
    const hero_layer_acts& A = s->acts[l];
    const hero_layer_grads& G = s->grads[l];
    const void* h_in = (l == 0) ? s->x : s->acts[l - 1].out;
    const bool hd = s->hidden_drop_threshold != 0u;
    HERO_REQUIRE(A.pre != nullptr, "stack bwd: layer %d has no saved FFN pre-activation", l);
    const int par = l & 1;
    void *ds2 = ds2_[par], *ds2_d = ds2_d_[par], *ds1 = ds1_[par], *ds1_d = ds1_d_[par];
    void *dpre = dpre_[par], *dqkv = dqkv_[par];
    // scratch[par] was last read by the weight gradients of layer l + 2
    if (two_streams && done_recorded[par])
      HERO_CUDA_CHECK(cudaStreamWaitEvent(chain, side->done[par], 0));

    // LN2 backward: ds2 (residual branch) and its dropout-masked copy (FFN-down branch)
    hero_ln_args ln;
    ln_base(&ln, A.s2, W.ln2_g, nullptr, s->eps, M, H, A.mean2, A.rstd2);
    ln.dy = dy; ln.dx = ds2; ln.dgamma = G.dln2_g; ln.dbeta = G.dln2_b;
    ln.dbias = G.db2;   // bias gradient of the FFN-down Linear = column sums of the masked ds2
    void* g2 = ds2;
    if (hd) {
      ln.dx_drop = ds2_d;
      ln.drop2_threshold = s->hidden_drop_threshold;
      ln.drop2_key = site_key(s->drop_key, l, 2);
      ln.drop2_scale = s->hidden_drop_scale;
      g2 = ds2_d;
    }
    HERO_STEP(ABL_LN_BWD, hero_ln_bwd(&ln, stream));
    HERO_TRY(publish());
    // FFN down
    HERO_STEP(ABL_WGRAD, Gemm(g2, H, 1, A.f, I, 1, H, I, M, G.dw2, I).f32_accumulate().run(wstream));
    // (its epilogue also accumulates the column sums of dpre = the FFN-up bias gradient)
    HERO_STEP(ABL_DGRAD, Gemm(g2, H, 0, W.w2, I, 1, M, I, H, dpre, I).act(ACT_GELU_GRAD).aux_in(A.pre, I).colsum(G.db1).run(stream));
    HERO_TRY(publish());
    // FFN up
    HERO_STEP(ABL_WGRAD, Gemm(dpre, I, 1, A.a, H, 1, I, H, M, G.dw1, H).f32_accumulate().run(wstream));
    HERO_STEP(ABL_DGRAD, Gemm(dpre, I, 0, W.w1, H, 1, M, H, I, da, H).resid(ds2, H).run(stream));
    // LN1 backward
    ln_base(&ln, A.s1, W.ln1_g, nullptr, s->eps, M, H, A.mean1, A.rstd1);
    ln.dy = da; ln.dx = ds1; ln.dgamma = G.dln1_g; ln.dbeta = G.dln1_b;
    ln.dbias = G.dbo;
    void* g1 = ds1;
    if (hd) {
      ln.dx_drop = ds1_d;
      ln.drop2_threshold = s->hidden_drop_threshold;
      ln.drop2_key = site_key(s->drop_key, l, 1);
      ln.drop2_scale = s->hidden_drop_scale;
      g1 = ds1_d;
    }
    HERO_STEP(ABL_LN_BWD, hero_ln_bwd(&ln, stream));
    HERO_TRY(publish());
    // attention output projection
    HERO_STEP(ABL_WGRAD, Gemm(g1, H, 1, A.cx, H, 1, H, H, M, G.dwo, H).f32_accumulate().run(wstream));
    HERO_STEP(ABL_DGRAD, Gemm(g1, H, 0, W.wo, H, 1, M, H, H, dcx, H).run(stream));
    // attention core
    HERO_STEP(ABL_ATTN_BWD, hero_attn_bwd(A.qkv, s->tile_tok0, s->tile_ntok, s->seq_lo, s->seq_hi, A.cx, dcx, A.lse,
                           dqkv, G.dbqkv, M, s->n_tiles, s->n_long, s->max_long, s->heads, 64, scale,
                           s->attn_drop_threshold,
                           site_key(s->drop_key, l, 0), s->attn_drop_scale, stream));
    HERO_TRY(publish());
    // QKV projection
    HERO_STEP(ABL_WGRAD, Gemm(dqkv, 3 * H, 1, h_in, H, 1, 3 * H, H, M, G.dwqkv, H).f32_accumulate().run(wstream));
    if (two_streams) {
      HERO_CUDA_CHECK(cudaEventRecord(side->done[par], side->stream));
      done_recorded[par] = true;
    }
    void* dx = (l == 0 && s->dx) ? s->dx : ((l & 1) ? dxa : dxb);
    if (l > 0 || s->dx)
      HERO_STEP(ABL_DGRAD, Gemm(dqkv, 3 * H, 0, W.wqkv, H, 1, M, H, 3 * H, dx, H).resid(ds1, H).run(stream));
    dy = dx;
  }
  if (two_streams && s->n_layers > 0) {   // every gradient is complete in `stream` order on return
    HERO_CUDA_CHECK(cudaEventRecord(side->joined, side->stream));
    HERO_CUDA_CHECK(cudaStreamWaitEvent(chain, side->joined, 0));
  }
  return HERO_OK;
}
