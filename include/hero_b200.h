/*
 * hero_b200 C-ABI — the drop-in boundary of the B200-native HERO encoder hot path.
 *
 * The reference (linjieli222/HERO) has no FFI layer: its boundary is the Python nn.Module
 * surface of model/{layers,embed,encoder,model}.py. Each entry point below replaces the device
 * arithmetic of one reference call site (cited per function, file:line relative to the reference
 * repo). They are what a ctypes binding on the reference side binds (see INTEGRATION.md).
 *
 * Conventions
 *   - plain C types only: device pointers, sizes, strides in ELEMENTS unless a name says bytes.
 *   - every function enqueues work on `stream` (a cudaStream_t passed as void*) and returns 0 on
 *     success or a non-zero hero_status; hero_last_error() describes the last failure of the
 *     calling thread. No hidden allocation; global state is limited to cached device
 *     attributes, the TMA descriptor encode entry point, the optional SM limit, and the layer
 *     runtime's second stream + events per device (hero_bert_stack_bwd, always joined into the
 *     caller's stream before the call returns).
 *   - "bf16" buffers are raw uint16 bfloat16; "f32" are float.
 *   - token-major packed layout: activations are [n_tokens, hidden] with only VALID (unmasked)
 *     tokens present; sequences are described by cu_seqlens[n_seq + 1] (int32 prefix sums).
 */
#ifndef HERO_B200_H_
#define HERO_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum hero_status {
  HERO_OK = 0,
  HERO_ERR_INVALID = 1, /* bad argument / unsupported shape */
  HERO_ERR_CUDA = 2,    /* CUDA runtime / driver error */
  HERO_ERR_NO_DEVICE = 3
} hero_status;

/* Library / device info. */
const char* hero_last_error(void);
int hero_version(void);
/* Returns SM count of the current device (148 on B200) or a negative hero_status. */
int hero_sm_count(void);

/* ------------------------------------------------------------------------------------------
 * GEMM family (tcgen05 / TMEM / TMA).   D[M,N] = epilogue( A · B^T-like contraction )
 *
 * Replaces every nn.Linear on the path — model/layers.py:125-127 (Q,K,V), :176 (attn out),
 * :237 (FFN up + gelu :16-25), :251 (FFN down), model/embed.py:112 (img_linear),
 * model/layers.py:82,90 (frame_transform Linear) — and their autograd backward
 * (dgrad: dX = dY·W, wgrad: dW = dYᵀ·X).
 *
 * Operand addressing (bf16):
 *   a_mn_major = 0 : A is [M, K] row-major, leading dim lda      (K contiguous)
 *   a_mn_major = 1 : A is stored as [K, M] row-major, lda        (M contiguous; "transposed")
 *   b_mn_major = 0 : B is [N, K] row-major, ldb                  (K contiguous; nn.Linear.weight)
 *   b_mn_major = 1 : B is stored as [K, N] row-major, ldb        (N contiguous)
 *   forward  Y = X·Wᵀ      : A = X  (0), B = W  (0)
 *   dgrad    dX = dY·W     : A = dY (0), B = W  (1)   [W is [N_out, K_in] = [K', N']]
 *   wgrad    dW = dYᵀ·X    : A = dY (1), B = X  (1), out_f32_accumulate = 1
 * Epilogue, applied in this order on v = acc:
 *   v += bias[n]                                  (bias != NULL; fp32)
 *   act: 0 none | 1 gelu_erf(v) | 2 relu(v) | 3 v * aux_in[m,n] | 4, 5 fused LM-head cross entropy
 *        (see the ce_* fields)
 *   if aux_out (what the backward needs of the activation):
 *        act 1: aux_out[m,n] = bf16(gelu_erf'(v))   (consumed by act 3 in the dgrad GEMM)
 *        else : aux_out[m,n] = bf16(v)              (pre-activation; ReLU backward uses its sign)
 *   dropout: v = keep(m*N+n) ? v * drop_scale : 0 (drop_threshold != 0; keep iff hash>=threshold)
 *   v += resid[m,n]                               (resid != NULL; bf16, or fp32 when resid_f32)
 *   out: bf16 store, fp32 store (out_f32_store: the pre-LayerNorm sums of the transformer layers
 *        stay fp32 end to end, like the fp32 residual stream of the reference under autocast), or
 *        fp32 atomic accumulate (out_f32_accumulate; split-K allowed)
 * Residual / saved-derivative tiles reach the epilogue by TMA (one 32-row slab per epilogue warp,
 * prefetched one slab ahead), outputs leave through double-buffered smem slabs and TMA stores.
 * Constraints: K % 8 == 0, N % 8 == 0, lds % 8 == 0, 16-byte aligned pointers; MN-major operands
 * need their contiguous extent to be a multiple of 64.
 * ---------------------------------------------------------------------------------------- */
typedef struct hero_gemm_args {
  const void* a; /* bf16 */
  const void* b; /* bf16 */
  int64_t lda, ldb;
  int32_t a_mn_major, b_mn_major;
  int32_t m, n, k;
  const float* bias;     /* [n] or NULL */
  const void* resid;     /* bf16 [m, ld_resid] or NULL */
  int64_t ld_resid;
  const void* aux_in;    /* bf16 [m, ld_aux_in], required for act == 3 (saved derivative) */
  int64_t ld_aux_in;
  void* aux_out;         /* bf16 [m, ld_aux_out] or NULL */
  int64_t ld_aux_out;
  void* out;             /* bf16 [m, ld_out] or f32 [m, ld_out] */
  int64_t ld_out;
  int32_t act;
  int32_t out_f32_accumulate;
  uint32_t drop_threshold; /* 0 = no dropout; else p * 2^32 */
  uint32_t drop_key;
  float drop_scale;        /* 1 / (1 - p) */
  int32_t block_n;         /* 0 = auto, else 128 or 256 */
  int32_t k_splits;        /* 0 = auto (only > 1 when out_f32_accumulate) */
  int32_t cta_pair;        /* 0 = auto, 1 = single-CTA tiles, 2 = force CTA pairs (cta_group::2,
                              256 x 256 tiles; needs block_n 256) */
  int32_t resid_f32;       /* resid is f32 [m, ld_resid] (needs out_f32_store) */
  int32_t out_f32_store;   /* out is f32 [m, ld_out], plain store (act 0 only; ld_out % 4 == 0) */
  /* Split-bf16 operands (both or neither; same layout / leading dims as a, b): the contraction
   * becomes a*b + a_lo*b + a*b_lo in ONE accumulator, i.e. operands with ~16 mantissa bits
   * (x_lo = bf16(x - float(bf16(x)))). Used for the frame_transform Linear (model/layers.py:86-93):
   * its ReLU gate flips on ~0.08 % of the units when the pre-activation is computed from plain
   * bf16 operands, which alone costs 4e-2 relative error in that layer's gradients. */
  const void* a_lo;
  const void* b_lo;
  /* LayerNorm-form residual (all four or none; needs resid_f32): the value added is
   *   (resid[m,n] - resid_ln_mean[m]) * resid_ln_rstd[m] * resid_ln_gamma[n] + resid_ln_beta[n],
   * i.e. LayerNorm(resid) in fp32, recomputed here from the pre-LayerNorm sum and the statistics
   * the LayerNorm kernel saved — the residual stream then needs no fp32 copy of LayerNorm outputs. */
  const float* resid_ln_mean;
  const float* resid_ln_rstd;
  const float* resid_ln_gamma;
  const float* resid_ln_beta;
  /* Fused LM-head cross entropy (act 4 forward, act 5 backward; MLM task, model/layers.py:330-354
   * + model/encoder.py:370-372). v = a . b^T + bias are the vocabulary logits of m masked tokens;
   * columns >= ce_n_valid (vocabulary padding, model/encoder.py:226-235) are excluded.
   *   act 4: no tile is stored (out may be NULL). For every 64-column slab t of row r:
   *          ce_partial[t * ce_ld_partial + r] = (max_j v_j, sum_j exp(v_j - max)) as float2 and
   *          ce_label_logit[r] = v[ce_label[r]]. hero_ce_finish turns them into loss + lse.
   *   act 5: out[r, c] = bf16( ce_grad[r] * (exp(v - ce_lse[r]) - [c == ce_label[r]]) ), 0 in the
   *          padding columns: d loss / d logits, ready for the dgrad / wgrad GEMMs. */
  const int32_t* ce_label;
  void* ce_partial;
  float* ce_label_logit;
  const float* ce_lse;
  const float* ce_grad;
  int64_t ce_ld_partial;
  int32_t ce_n_valid;
  /* Optional, bf16 stores only: f32 [n]; the column sums of the (bf16-rounded) output rows < m
   * are ACCUMULATED into it from the epilogue's staged slabs. With `out` = the gradient of a
   * Linear's output this is that Linear's bias gradient, for free instead of a second pass over
   * `out` (the FFN-up bias gradient of model/layers.py:210-225 comes from the x gelu' dgrad). */
  float* out_colsum;
} hero_gemm_args;

int hero_gemm_bf16(const hero_gemm_args* args, void* stream);

/* Measurement aid for the roofline line of bench.py: between begin and end every GEMM launch (direct
 * or issued by the layer runtime) is bracketed by CUDA events on its stream; end synchronises and
 * returns the summed kernel time [ms], the summed 2*M*N*K [FLOP] and the number of launches. */
int hero_gemm_profile_begin(void);
int hero_gemm_profile_end(double* ms, double* flops, int64_t* launches);

/* ------------------------------------------------------------------------------------------
 * Fused row kernels: gather + add + LayerNorm (+ dropout) + scatter. One entry point per
 * direction; the library picks the kernel (persistent register-resident fast path for plain bf16
 * rows of <= 768 columns incl. a one-pass backward with dgamma / dbeta / dbias, CTA-per-row kernel
 * for the 4352-wide rows, generic warp-per-row kernel otherwise).
 *
 * Replaces apex FusedLayerNorm and the embedding sums around it:
 *   model/layers.py:178,253      LN(dropout(dense(x)) + residual), eps 1e-12 (post-GEMM form:
 *                                x = pre-LN sum written by the GEMM epilogue)
 *   model/embed.py:44-58         LN(word[ids] + pos[pos_ids] + type[1]); dropout
 *                                (x = word table f32, x_rows = ids, add_tab = pos table,
 *                                 add_vec = type row)
 *   model/embed.py:108-116       img: x (+ mask_emb[mask]) -> LN_4352 ; then after img_linear
 *                                LN(proj + pos_img[k] + type[1]); dropout
 *   model/embed.py:156-160       LN(frame_feat + pos[t]); dropout
 *   model/layers.py:88-89        LinearLayer.LayerNorm over the 4352-d frame feature
 * Forward, for output row i in [0, n_rows):
 *   s = X[x_rows ? x_rows[i] : i]  (bf16 or f32, row length H)
 *       + (add_tab ? add_tab[add_idx[i]] : 0) + (add_vec ? add_vec : 0)
 *   y = (s - mean(s)) * rsqrt(var_biased(s) + eps) * gamma + beta      (fp32 statistics)
 *   y = dropout(y)  (element index i*H + j)  -> bf16 -> Y[y_rows ? y_rows[i] : i]
 *   mean[i], rstd[i] saved when non-NULL.
 * Backward recomputes s from the same gather description and returns
 *   dx[i] (bf16, grad wrt s), optional dx_drop[i] = dx[i] * mask2 * scale2 (the gradient that
 *   flows into the dropout'ed GEMM branch of a post-GEMM LN), fp32 atomic scatter-adds of dx into
 *   d_x_tab[x_rows[i]] / d_add_tab[add_idx[i]], and dgamma/dbeta (atomic accumulate per block).
 *   Rows whose x_rows / add_idx equal *_pad_idx get no table gradient (nn.Embedding padding_idx).
 *   Heavily shared tables (position / type rows) are better reduced with
 *   hero_gather_sum_rows_f32 / hero_colsum_bf16 over dx than with the atomic path.
 * Constraints: H % 8 == 0, H <= 4352.
 * ---------------------------------------------------------------------------------------- */
typedef struct hero_ln_args {
  /* gather description (shared by fwd and bwd) */
  const void* x;
  int32_t x_is_f32;
  const int32_t* x_rows;   /* NULL = identity */
  const float* add_tab;    /* NULL = none */
  const int32_t* add_idx;
  const float* add_vec;    /* NULL = none */
  const float* gamma;
  const float* beta;
  float eps;
  int32_t n_rows, h;
  /* forward outputs / backward saved stats */
  void* y;                 /* bf16 */
  void* y_lo;              /* optional bf16 remainder bf16(y_f32 - float(bf16 y)) at the same rows: the
                              low half of a split-bf16 GEMM operand (see hero_gemm_args.a_lo) */
  const int32_t* y_rows;   /* NULL = identity; also indexes dy in bwd */
  float* y_f32;            /* optional fp32 copy of y (same rows, after dropout): the residual
                              stream consumed by the next GEMM epilogue; NULL = none; h <= 768 */
  float* mean;
  float* rstd;
  /* dropout applied to the LN output */
  uint32_t drop_threshold, drop_key;
  float drop_scale;
  /* backward only */
  const void* dy;          /* bf16, indexed like y */
  void* dx;                /* bf16 [n_rows, h] or NULL */
  void* dx_drop;           /* bf16 [n_rows, h] or NULL */
  uint32_t drop2_threshold, drop2_key;
  float drop2_scale;
  float* d_x_tab;          /* f32 table grad (scatter by x_rows) or NULL */
  int32_t x_pad_idx;       /* -1 = none */
  float* d_add_tab;        /* f32 or NULL */
  int32_t add_pad_idx;     /* -1 = none */
  float* dgamma;           /* f32 [h] or NULL */
  float* dbeta;            /* f32 [h] or NULL */
  float* dbias;            /* f32 [h] or NULL: += column sums of dx_drop (dx when dx_drop is NULL),
                              i.e. the bias gradient of the Linear that fed this LayerNorm */
} hero_ln_args;

int hero_ln_fwd(const hero_ln_args* args, void* stream);
int hero_ln_bwd(const hero_ln_args* args, void* stream);

/* ------------------------------------------------------------------------------------------
 * Variable-length multi-head self-attention over packed sequences (tcgen05 / TMEM / TMA).
 *
 * Replaces model/layers.py:129-160 (transpose_for_scores, QK^T/sqrt(d) + additive -10000 key
 * mask, softmax, dropout on probabilities, P·V, head merge) and its backward. Only valid tokens
 * exist in the packed layout, so the key-padding mask of model/layers.py:299-302 becomes "a row
 * attends to the tokens of its own sequence".
 *   qkv   bf16 [n_tok, 3*heads*64]  (Q | K | V, each head-major inside)
 *   ctx   bf16 [n_tok, heads*64]
 *   lse   f32  [n_tok, heads]  log2-domain log-sum-exp of the scaled scores of each (token, head)
 *                              row; written by the forward (may be NULL in inference), read by the
 *                              backward, which rebuilds the probabilities in one pass
 * Host-built plan (int32, device memory; hero_b200/plan.py SeqPlan):
 *   tile_tok0[n_tiles], tile_ntok[n_tiles]  consecutive sequences grouped into tiles of <= 128
 *                                           tokens and <= 16 sequences; a sequence never
 *                                           straddles two tiles
 *   seq_lo[n_tok], seq_hi[n_tok]            [lo, hi) packed-token range of each token's sequence
 * One CTA per (tile, head): S = QK^T and O = PV (forward), S, dP, dQ, dK, dV (backward) are
 * tcgen05.mma contractions with fp32 accumulators in TMEM; probabilities never reach HBM.
 * The "own sequence only" mask is itself a tensor-core product: one extra K = 16 step adds 16384
 * to every same-sequence (query, key) score (membership matrix x its transpose), which leaves the
 * row's softmax unchanged and sends every other column's exp2 to exactly 0 - no per-element
 * compares in the softmax loops (hence the 16-sequence limit per tile).
 * Dropout: one 32-bit counter hash per (token i, head h, group of 8 tile columns), index
 * ((i*heads + h)*128 + group); its four pair-words (the hash and three multiply-xorshift
 * derivations) give 15 bits per probability; forward and backward regenerate the same words
 * from the same plan.
 * The backward takes the saved forward output (D_i = dO_i . O_i). With `dbias` != NULL it also
 * ACCUMULATES the column sums of dqkv (= the bias gradient of the QKV projection, f32 [3*H])
 * into it, through one more MMA over the staged dQ/dK/dV tiles.
 * Sequences of more than 128 tokens (up to 768; the reference's position table allows 514) take
 * the LAST n_long tiles of the plan, one whole sequence per tile (tile_ntok = its length,
 * max_long = the longest): they run on fp32 CUDA-core kernels with the same arithmetic contract
 * (one CTA per (sequence, head), K / V or Q / dO staged in shared memory).
 * Constraints: head_dim == 64, sequences <= 768 tokens.
 * ---------------------------------------------------------------------------------------- */
int hero_attn_fwd(const void* qkv, const int32_t* tile_tok0, const int32_t* tile_ntok,
                  const int32_t* seq_lo, const int32_t* seq_hi, void* ctx, float* lse,
                  int32_t n_tok, int32_t n_tiles, int32_t n_long, int32_t max_long, int32_t heads,
                  int32_t head_dim, float scale, uint32_t drop_threshold, uint32_t drop_key,
                  float drop_scale, void* stream);
int hero_attn_bwd(const void* qkv, const int32_t* tile_tok0, const int32_t* tile_ntok,
                  const int32_t* seq_lo, const int32_t* seq_hi, const void* ctx, const void* dctx,
                  const float* lse, void* dqkv, float* dbias, int32_t n_tok, int32_t n_tiles,
                  int32_t n_long, int32_t max_long, int32_t heads, int32_t head_dim, float scale,
                  uint32_t drop_threshold, uint32_t drop_key, float drop_scale, void* stream);

/* ------------------------------------------------------------------------------------------
 * Native layer runtime: a whole stack of BertLayers (model/layers.py:257-327) forward / backward
 * per call. The reference dispatches ~50 PyTorch ops per layer from Python; even one ctypes call
 * per kernel left the host as the bottleneck (11 ms of launches per 15 ms step), so the per-layer
 * launch sequence lives here:
 *   forward   qkv = x Wqkv^T + b -> attention -> s1 = drop(ctx Wo^T + bo) + x -> a = LN(s1) ->
 *             f = gelu(a W1^T + b1) (pre-activation kept when `pre` != NULL) ->
 *             s2 = drop(f W2^T + b2) + a -> out = LN(s2)
 *             The residual stream (x, s1, a, s2, out) is carried in FP32 — the GEMM epilogues add
 *             an fp32 residual and store fp32 sums, the LayerNorm kernels read them and write a
 *             bf16 copy (next GEMM operand) plus an fp32 copy (next residual) — exactly where
 *             torch.autocast(bfloat16) keeps fp32 in the reference; only GEMM operands are bf16.
 *   backward  the exact adjoint chain (LN bwd with fused dropout-masked copy, bias column sums,
 *             split-K wgrads accumulated in fp32 into `grads`, dgrads with fused GELU' / residual
 *             adds, attention backward)
 * All buffers are caller-owned device memory; `weights`, `acts`, `grads` are HOST arrays of
 * n_layers entries. Gradients are ACCUMULATED (+=) into `grads` (point them at zeroed memory or
 * at the existing .grad buffers). Dropout keys derive from (drop_key, layer, site), identically in
 * forward and backward; thresholds of 0 disable dropout.
 * ---------------------------------------------------------------------------------------- */
typedef struct hero_layer_weights {
  const void* wqkv;  /* bf16 [3H, H] (query | key | value rows) */
  const float* bqkv; /* [3H] */
  const void* wo;    /* bf16 [H, H] */
  const float* bo;
  const float* ln1_g;
  const float* ln1_b;
  const void* w1;    /* bf16 [I, H] */
  const float* b1;
  const void* w2;    /* bf16 [H, I] */
  const float* b2;
  const float* ln2_g;
  const float* ln2_b;
} hero_layer_weights;

typedef struct hero_layer_acts { /* bf16 unless noted; [n_tok, ...] */
  void* qkv;    /* [n_tok, 3H] */
  void* cx;     /* attention output [n_tok, H] */
  float* lse;   /* f32 [n_tok, heads]: attention log-sum-exp (NULL in inference) */
  float* s1;    /* f32 pre-LN sum after the attention block */
  float* mean1;
  float* rstd1;
  void* a;      /* LN(s1), bf16: operand of the FFN-up GEMM and of its weight gradient */
  float* a_f32; /* unused (NULL): the FFN-down epilogue recomputes LN(s1) in fp32 from s1, mean1,
                   rstd1 and the LayerNorm parameters (hero_gemm_args.resid_ln_*) */
  void* pre;    /* gelu'(FFN pre-activation) [n_tok, I], saved for the backward; NULL in inference */
  void* f;      /* gelu(pre) [n_tok, I] */
  float* s2;    /* f32 pre-LN sum after the FFN */
  float* mean2;
  float* rstd2;
  void* out;    /* LN(s2), bf16: the layer output as the next layer's GEMM operand */
  float* out_f32; /* LN(s2), f32: written only when non-NULL (the caller wants the stack's result in
                     fp32: last layer); the next layer's residual is recomputed from s2 */
} hero_layer_acts;

typedef struct hero_layer_grads { /* fp32, accumulated */
  float* dwqkv; float* dbqkv; float* dwo; float* dbo; float* dln1_g; float* dln1_b;
  float* dw1; float* db1; float* dw2; float* db2; float* dln2_g; float* dln2_b;
} hero_layer_grads;

typedef struct hero_stack_args {
  int32_t n_layers, n_tok, hidden, inter, heads, n_tiles;
  int32_t n_long, max_long;      /* long-sequence tiles of the attention plan (see hero_attn_fwd) */
  float eps;
  const hero_layer_weights* weights;
  const hero_layer_acts* acts;
  const hero_layer_grads* grads; /* backward only */
  const void* x;                 /* stack input, bf16 [n_tok, H] */
  const float* x_f32;            /* the same input in f32 (residual of layer 0); forward only */
  const int32_t* tile_tok0;      /* attention plan, see hero_attn_fwd */
  const int32_t* tile_ntok;
  const int32_t* seq_lo;
  const int32_t* seq_hi;
  uint32_t hidden_drop_threshold, attn_drop_threshold, drop_key;
  float hidden_drop_scale, attn_drop_scale;
  /* backward only */
  const void* dout;              /* bf16 [n_tok, H] gradient of the last layer's output */
  void* dx;                      /* bf16 [n_tok, H] gradient of x (may be NULL for no input grad) */
  void* scratch;                 /* >= hero_bert_stack_bwd_scratch_bytes(...) bytes */
} hero_stack_args;

int hero_bert_stack_fwd(const hero_stack_args* args, void* stream);
int hero_bert_stack_bwd(const hero_stack_args* args, void* stream);
int64_t hero_bert_stack_bwd_scratch_bytes(int32_t n_tok, int32_t hidden, int32_t inter);

/* ------------------------------------------------------------------------------------------
 * Row utilities (HBM-bound).
 * ---------------------------------------------------------------------------------------- */
/* dst[i] = bf16(src[i]); keeps bf16 working copies of the fp32 master weights. */
int hero_cast_f32_to_bf16(const float* src, void* dst, int64_t n, void* stream);
/* dst[i, :] = idx[i] >= 0 ? src[idx[i], :] : 0   (bf16 rows of length h, h % 8 == 0).
 * Packs/unpacks padded <-> packed token layouts (replaces torch.gather at
 * model/encoder.py:271-279) and is the backward of hero_gather_sum_rows_bf16. */
int hero_gather_rows_bf16(const void* src, const int32_t* idx, void* dst, int32_t n, int32_t h,
                          void* stream);
/* dst[i, :] = sum_{e in [off[i], off[i+1])} src[idx[e], :]   (CSR gather-sum, fp32 accumulate).
 * Deterministic replacement of collect_frame_outputs (model/model.py:156-187). */
int hero_gather_sum_rows_bf16(const void* src, const int32_t* off, const int32_t* idx, void* dst,
                              int32_t n, int32_t h, void* stream);
/* dst[i, :] = idx[i] >= 0 ? src[idx[i], :] : 0 over f32 rows (h % 4 == 0): unpacks the f32 layer
 * output of the last transformer layer into the padded (B, T, H) / (N, L, H) API tensors. */
int hero_gather_rows_f32(const float* src, const int32_t* idx, float* dst, int32_t n, int32_t h,
                         void* stream);
/* Same CSR gather-sum over bf16 rows but accumulating into fp32 rows: dst[i, :] += sum(...).
 * Deterministic embedding-table gradients (position tables) from the LN backward's dx. */
int hero_gather_sum_rows_f32(const void* src, const int32_t* off, const int32_t* idx, float* dst,
                             int32_t n, int32_t h, void* stream);
/* out[n] += sum_m x[m, n]  (bias gradients). */
int hero_colsum_bf16(const void* x, int64_t ld, int32_t m, int32_t n, float* out, void* stream);
/* out = dy * (pre > 0)   (ReLU backward of model/layers.py:92). */
int hero_relu_bwd_bf16(const void* dy, const void* pre, void* out, int64_t n, void* stream);

/* ------------------------------------------------------------------------------------------
 * Optimizer (flat buffers). Follows optim/adamw.py:80-104 exactly:
 *   g' = g * grad_scale
 *   m = b1*m + (1-b1)*g' ; v = b2*v + (1-b2)*g'^2
 *   p -= step_size * m / (sqrt(v) + eps)      step_size = lr*sqrt(1-b2^t)/(1-b1^t) (host-computed)
 *   p -= lr_wd * p                            lr_wd = lr * weight_decay (0 for bias/LayerNorm)
 * and optionally refreshes the bf16 working copy.
 * ---------------------------------------------------------------------------------------- */
int hero_adamw_step(float* p, const float* g, float* m, float* v, void* p_bf16, int64_t n,
                    float step_size, float beta1, float beta2, float eps, float lr_wd,
                    float grad_scale, const float* clip_sumsq, float clip_max_norm, void* stream);
/* clip_sumsq != NULL folds global-norm clipping (train_vcmr.py:258-259) into the update without a
 * device->host round trip: g' is additionally scaled by min(1, clip_max_norm / (sqrt(*clip_sumsq)
 * + 1e-6)), *clip_sumsq being the device scalar accumulated by hero_sumsq_f32 over ALL gradients. */
/* Combines the per-slab partials of an act-4 GEMM: lse[r] = log sum_c exp(v[r, c]) and
 * loss[r] = lse[r] - label_logit[r] (F.cross_entropy, reduction='none'), r < m. */
int hero_ce_finish(const void* ce_partial, int64_t ld_partial, int32_t n_slabs,
                   const float* label_logit, int32_t m, float* loss, float* lse, void* stream);
/* out[0] += sum x^2 (global-norm clipping, train_vcmr.py:258-259). */
int hero_sumsq_f32(const float* x, int64_t n, float* out, void* stream);

/* ------------------------------------------------------------------------------------------
 * Video-subtitle matching / moment-retrieval head (SURVEY.md §8f rank 1): the ops that follow the
 * encoder in HeroForPretraining / HeroForVcmr.
 *   model/pretrain.py:364-413  get_video_level_scores: F.normalize (eps 1e-5) of queries and
 *       frames, einsum("md,nld->mln"), mask_logits, max over frames
 *   model/pretrain.py:128-166  _get_st_ed_prob (non-cross form): einsum("bd,bld->bl"), two
 *       Conv1d(1, 1, k, padding k/2, bias=False), mask_logits
 * ---------------------------------------------------------------------------------------- */
/* x^[r] = x[r] / max(|x[r]|_2, eps) written as split-bf16 halves hi + lo (operands of a split-bf16
 * hero_gemm_bf16, ~16 mantissa bits); inv_norm[r] = 1 / max(|x[r]|, eps), NEGATED where the clamp
 * was active. d % 4 == 0. */
int hero_l2norm_split_f32(const float* x, int64_t rows, int32_t d, float eps, void* hi, void* lo,
                          float* inv_norm, void* stream);
/* scores[m, n] = max_l (mask[n, l] ? s[m, n * len + l] : -1e4), argmax[m, n] = its (lowest) l;
 * s is the [nq, ld_s] fp32 output of the q^ . c^ GEMM, mask [nv, len] bytes. */
int hero_vsm_masked_max(const float* s, int64_t ld_s, const uint8_t* mask, int32_t nq, int32_t nv,
                        int32_t len, float* scores, int32_t* argmax, void* stream);
/* Backward of the three steps above given g = d loss / d scores [nq, nv]: dq [nq, d] and
 * dctx [nv * len, d] (fp32, OVERWRITTEN; either may be NULL), through the max (gradient to the
 * arg-max frame only, none through masked frames) and the normalisations. d <= 1024. */
int hero_vsm_scores_bwd(const float* g, const int32_t* argmax, const uint8_t* mask, const void* q_hi,
                        const void* q_lo, const float* q_inv, const void* c_hi, const void* c_lo,
                        const float* c_inv, int32_t nq, int32_t nv, int32_t len, int32_t d,
                        float* dq, float* dctx, void* stream);
/* Span logits of n (query, clip) pairs: sim[b, l] = query[b] . ctx[b, l];
 * st / ed[b, l] = mask ? sum_k w[k] * sim[b, l + k - K/2] : -1e4 (zero padding). len <= 512,
 * odd K <= 15, d % 4 == 0. The backward OVERWRITES dquery [n, d], dctx [n, len, d] and
 * ACCUMULATES (+=) dw_st / dw_ed [K]. */
int hero_vsm_span_fwd(const float* query, const float* ctx, const uint8_t* mask, const float* w_st,
                      const float* w_ed, int32_t n, int32_t len, int32_t d, int32_t k, float* sim,
                      float* st, float* ed, void* stream);
int hero_vsm_span_bwd(const float* dst, const float* ded, const uint8_t* mask, const float* w_st,
                      const float* w_ed, const float* sim, const float* query, const float* ctx,
                      int32_t n, int32_t len, int32_t d, int32_t k, float* dquery, float* dctx,
                      float* dw_st, float* dw_ed, void* stream);

/* ------------------------------------------------------------------------------------------
 * Video question answering head (TVQA / How2QA): HeroForVideoQA.get_modularized_video,
 * model/videoQA.py:36-59, on the packed fp32 output y [n_joint, h] of the query-fused temporal
 * stack (model/videoQA.py:66-82). frame_tok [nv * nq * t] is the row of y holding frame t of
 * answer candidate q of question v, or -1 at a padded frame (x = 0 there). With x = y[frame_tok]:
 *   s_se = w_se . x, s_qa = w_qa . x; score where valid, exactly -1e4 where not (mask_logits)
 *   a_se = softmax over q (videoQA.py:45-47), a_qa = softmax over t (videoQA.py:48-50)
 *   p_se [nv, t, h] = sum_q a_se x (videoQA.py:52-54), p_qa [nv, nq, h] = sum_t a_qa x (:55-57)
 * s_se / s_qa / a_se / a_qa are [nv, nq, t] fp32 (the a_* feed the backward). nq <= 64,
 * t <= 1024, h % 4 == 0. Two kernel launches. */
int hero_videoqa_pool_fwd(const float* y, const int32_t* frame_tok, const float* w_se,
                          const float* w_qa, int32_t nv, int32_t nq, int32_t t, int32_t h,
                          float* s_se, float* s_qa, float* a_se, float* a_qa, float* p_se,
                          float* p_qa, void* stream);
/* Backward given dp_se / dp_qa: dy [n_joint, h] receives d loss / dx at every frame row
 * (OVERWRITTEN there; other rows, the QA tokens sliced off at model/videoQA.py:82, are not
 * touched: zero them first); dw_se / dw_qa [h] are ACCUMULATED (+=). The softmax Jacobian terms
 * are zero at padded frames. da_se / da_qa: [nv, nq, t] fp32 scratch. Two kernel launches. */
int hero_videoqa_pool_bwd(const float* y, const int32_t* frame_tok, const float* w_se,
                          const float* w_qa, const float* a_se, const float* a_qa,
                          const float* dp_se, const float* dp_qa, int32_t nv, int32_t nq,
                          int32_t t, int32_t h, float* da_se, float* da_qa, float* dy,
                          float* dw_se, float* dw_qa, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HERO_B200_H_ */
