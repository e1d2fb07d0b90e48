/*
 * dalle_b200.h — C ABI of libdalle_b200.so, the B200 (sm_100a) hot path of the DALL-E transformer block.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  Every entry point replaces an op sequence that the
 * reference (lucidrains/DALLE-pytorch, /root/reference/dalle_pytorch/) evaluates with aten calls; the
 * reference file:line each one stands in for is cited next to its declaration.  The host side
 * (the .py files of dalle_pytorch_b200/) mirrors the reference's module API and calls these functions through ctypes.
 *
 * Conventions
 *   - plain C: POD parameter structs of raw DEVICE pointers, sizes and flags; no torch types.
 *   - the library never allocates, frees or retains device memory; the caller owns every buffer.
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued asynchronously on it.
 *   - return 0 on success, a negative db200_status on failure; dalle_b200_last_error() returns a
 *     thread-local message.  No exceptions cross the ABI and nothing aborts.
 *   - re-entrant: forward is called from the Python thread, backward from autograd's device thread.
 *   - dtype: DB200_F32 computes and stores in fp32 (parity mode, tolerance rtol 1e-3 / atol 1e-5 against
 *     the reference CPU path); DB200_BF16 stores activations/weights in bf16 with fp32 accumulation
 *     (speed mode: tcgen05 tensor-core GEMMs).  The residual stream, LayerNorm statistics, softmax
 *     statistics and all parameter gradients are always fp32.
 */
#ifndef DALLE_B200_H
#define DALLE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DALLE_B200_VERSION 112

typedef enum {
  DB200_OK = 0,
  DB200_ERR_BAD_ARG = -1,      /* shape / pointer / flag combination not supported */
  DB200_ERR_UNSUPPORTED = -2,  /* valid request the kernels do not implement (e.g. dim_head != 64) */
  DB200_ERR_CUDA = -3,         /* CUDA runtime / driver error at launch */
  DB200_ERR_NO_DEVICE = -4     /* no sm_100 device / driver entry point missing */
} db200_status;

typedef enum { DB200_F32 = 0, DB200_BF16 = 1 } db200_dtype;

/* attention sparsity pattern = allowed(query i, key j) predicate evaluated inside the kernels */
typedef enum {
  DB200_ATTN_FULL = 0,      /* Attention                    attention.py:39-99   (causal triu or none)        */
  DB200_ATTN_AXIAL_ROW = 1, /* SparseAxialCausalAttention   attention.py:225-335 axis=0                       */
  DB200_ATTN_AXIAL_COL = 2, /*                              axis=1                                             */
  DB200_ATTN_CONV_LIKE = 3, /* SparseConvCausalAttention    attention.py:103-221                              */
  DB200_ATTN_STATIC = 4     /* Attention(static_mask=...)   attention.py:89-90 ; transformer.py:333-350       */
} db200_attn_pattern;

typedef enum {
  DB200_EPI_STORE = 0,     /* C = acc (+bias)                                       nn.Linear                  */
  DB200_EPI_QKV = 1,       /* head split + rotary(q,k,v) + q*scale                  attention.py:63-69,263-269 */
  DB200_EPI_RESID = 2,     /* out = resid + sign*scale*(acc+bias)                   attention.py:97 / transformer.py:118,88 ; reversible.py:139-140 */
  DB200_EPI_GEGLU = 3,     /* h = (a+ba) * gelu_erf(g+bg), also stores u=[a|g]      transformer.py:106-109,115 */
  DB200_EPI_GEGLU_BWD = 4  /* du = [dh*gelu(g) | dh*a*gelu'(g)]                     autograd of the above      */
} db200_epilogue;

/* SMALLM: weight-streaming mma.sync kernel for 1 <= M <= 32 rows (decoding; M > 16 = a second 16-row A fragment, e.g. the 2b rows of
 * classifier-free guidance), bf16 K-major operands, K % 256 == 0, STORE / RESID / GEGLU;
 * chosen explicitly by the caller (AUTO never selects it), DB200_ERR_UNSUPPORTED when the problem does not qualify */
typedef enum { DB200_GEMM_AUTO = 0, DB200_GEMM_SIMT = 1, DB200_GEMM_TCGEN05 = 2, DB200_GEMM_SMALLM = 3 } db200_gemm_backend;

int dalle_b200_version(void);
const char* dalle_b200_last_error(void);
/* 1 if device `dev` is an sm_100 part on which the tcgen05/TMA kernels can run, else 0 */
int dalle_b200_device_ok(int dev);
/* sizeof() of the parameter structs in declaration order (ln_shift_fwd, ln_shift_bwd, gemm, attn_fwd, attn_bwd,
 * scale_bwd) so that a foreign-language binding can verify its struct layout at load time; returns the count */
int dalle_b200_abi_sizes(int* out, int capacity);

/* ---------------------------------------------------------------------------------------------
 * LayerNorm (+ token shift) producing the GEMM A operand.
 * Replaces PreNorm.norm + PreShiftToken.forward: transformer.py:100, 155-186 (training branch).
 * x [rows = batch*n, d] fp32 (residual stream) -> out [rows, d] (dtype), mean/rstd [rows] fp32 saved
 * for backward.  do_ln=0: plain copy/cast; do_shift=0: no shift (shift_tokens=False or n < text_len).
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  int batch, n, d;
  int text_len, fmap;       /* text_len = text_seq_len + 1 (<bos>), fmap = image_fmap_size */
  int do_ln, do_shift;
  int out_dtype;
  float eps;
  const float* x;
  const float* gamma;
  const float* beta;
  void* out;
  float* mean;
  float* rstd;
} db200_ln_shift_fwd_params;
int dalle_b200_ln_shift_fwd(const db200_ln_shift_fwd_params* p, void* stream);

/* backward of the above: dx = dres + LN_bwd(unshift(d_out)); dgamma/dbeta are ACCUMULATED (+=) */
typedef struct {
  int batch, n, d;
  int text_len, fmap;
  int do_ln, do_shift;
  int dout_dtype;
  const void* d_out;        /* [rows, d] gradient w.r.t. the shifted LN output (dtype) */
  const float* x;
  const float* mean;
  const float* rstd;
  const float* gamma;
  const float* dres;        /* optional fp32 [rows, d] added to the result (the residual branch) */
  float* dx;                /* [rows, d] fp32 */
  float* dgamma;            /* [d] fp32, += */
  float* dbeta;             /* [d] fp32, += */
  /* Optional fusion of the UPSTREAM sub-layer's LayerScale adjoint (what dalle_b200_scale_bwd would compute from this dx, which
   * is that sub-layer's output gradient) while dx is still in registers; saves re-reading dx.  d = 1024 only; up_dy == NULL = off.
   *   up_dy = up_sign * up_scale (.) dx  (dout_dtype);  up_dscale += up_sign * sum_rows dx (.) up_y;  up_dbias += sum_rows up_dy */
  const void* up_y;         /* [rows, d] (dout_dtype) upstream branch output, needed for up_dscale; may be NULL */
  const float* up_scale;    /* [d] fp32 or NULL (= 1) */
  float up_sign;
  void* up_dy;              /* [rows, d] (dout_dtype) out */
  float* up_dscale;         /* [d] fp32, += ; may be NULL */
  float* up_dbias;          /* [d] fp32, += ; may be NULL */
} db200_ln_shift_bwd_params;
int dalle_b200_ln_shift_bwd(const db200_ln_shift_bwd_params* p, void* stream);

/* ---------------------------------------------------------------------------------------------
 * GEMM with fused epilogue:  acc[M,N] = sum_k A(m,k) * B(n,k)
 *   a_mn_major = 0: A(m,k) = A[m*lda + k] (K-major)      1: A(m,k) = A[k*lda + m] (M-major)
 *   b_mn_major = 0: B(n,k) = B[n*ldb + k] (K-major)      1: B(n,k) = B[k*ldb + n] (N-major)
 * forward  Linear  : A = activations (K-major), B = weight [out,in] (K-major)      attention.py:63,97 transformer.py:114,118
 * dgrad            : A = dY (K-major), B = weight [out,in] read as (N=in, K=out) (N-major)
 * wgrad            : A = dY^T (M-major), B = X^T (N-major), C = dW [out,in] fp32
 * dtype selects fp32 (SIMT FFMA) or bf16 (tcgen05.mma kind::f16, TMA-fed) operands; accumulation fp32.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  int M, N, K;
  int dtype;                /* operand dtype of A and B */
  int backend;              /* db200_gemm_backend */
  const void* A; int64_t lda; int a_mn_major;
  const void* B; int64_t ldb; int b_mn_major;
  int epilogue;             /* db200_epilogue */
  /* STORE */
  void* C; int64_t ldc; int c_dtype; const float* bias;   /* bias [N] fp32 optional */
  int split_k_ok;           /* STORE, fp32 C, no bias: C is zero-initialised, the kernel may split K and reduce with fp32 atomics */
  void* C_multicast;        /* STORE, fp32, no bias, tcgen05 backend: if not NULL, c_scale * acc is ADDED into every GPU's copy of a
                               symmetric buffer through this NVLink multicast address (multimem.red, reduced in the NVSwitch) instead
                               of being stored to C -- the data-parallel gradient sum fused into the weight-gradient GEMM.  Same
                               [M, ldc] indexing as C, 16-byte aligned; the buffers must be zero before the first contribution. */
  float c_scale;            /* multicast mode only (e.g. 1 / world size) */
  /* QKV: N = 3*heads*dim_head; rows m = b*seq_n + p */
  void* q; void* k; void* v;                 /* [batch, heads, seq_n, dim_head] (dtype)                  */
  const float* cos_t; const float* sin_t;    /* [n_pos, dim_head/2] fp32, (1,0) on pass-through pairs; NULL = no rotary */
  int seq_n, heads, dim_head, pos_offset;
  float q_scale;
  /* RESID: out[m,n] = resid[m,n] + sign*scale[n]*(acc + bias[n]); y_out (dtype, optional) keeps acc+bias */
  const float* resid; const float* scale; float sign; void* y_out; float* out;
  /* GEGLU: N = 2*hidden; bias [2*hidden]; u_out [M, 2*hidden] (dtype, optional), h_out [M, hidden] (dtype) */
  void* u_out; void* h_out; int hidden;
  /* GEGLU_BWD: N = hidden; acc = dh; u_in [M, 2*hidden]; du_out [M, 2*hidden] (dtype) */
  const void* u_in; void* du_out;
} db200_gemm_params;
int dalle_b200_gemm(const db200_gemm_params* p, void* stream);
/* which backend dalle_b200_gemm would run for *p (DB200_GEMM_SIMT or DB200_GEMM_TCGEN05); no launch */
int dalle_b200_gemm_select(const db200_gemm_params* p);

/* ---------------------------------------------------------------------------------------------
 * Fused attention (flash-style, never materialises [n,n]) for every pattern of the reference.
 * q [batch, heads, n_q, 64], k,v [batch, heads, n_k, 64] with rotary and q-scale already applied (EPI_QKV);
 * queries are the LAST n_q positions of the n_k keys (n_q == n_k in training; n_q < n_k for cached decoding,
 * attention.py:71-76).
 * out [batch, n_q, heads*64] (merged heads, A operand of to_out), lse [batch, heads, n_q] fp32.
 * Replaces attention.py:78-96 and :271-331 (+ :147-207 for conv_like).
 *
 * gather != 0 (axial patterns, bf16, dim_head 64, fmap in {16,32,64}, n_q == n_k == n with n = text_len + fmap^2 [- 1], no
 * key mask): the kernels tile the TEXT keys and each group of 128 / fmap image lines separately and, for AXIAL_COL, fetch
 * the lines with strided TMA boxes (what attention.py:287-292 does with rearrange(..., axis = 1)).  Layout contract:
 *   q, k, v : [batch, heads, n_alloc, 64] with n_alloc = text_len + fmap^2, rows >= n ZERO (the reference pads the
 *             sequence with a zero token, attention.py:255-258; dalle_b200_qkv_rotary writes this layout);
 *   lse, delta : [batch, heads, n_stat] with n_stat = roundup(text_len, 64) + fmap^2 (library-internal ordering);
 *   d_out (backward, AXIAL_COL, n = text_len + fmap^2 - 1): one extra row of heads*64 elements must exist after the last
 *             token row; the library zeroes it.
 * Everything else (out, dqkv, the rotary tables) keeps the layouts documented here.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  int batch, heads, n_q, n_k, dim_head;
  int dtype;
  int pattern;              /* db200_attn_pattern */
  int causal;               /* FULL / STATIC only: apply j <= i (attention.py:84-87) */
  int stable;               /* stable_softmax (attention.py:27-30); alpha = 2^10 is an exact rescale, see DESIGN.md */
  int text_len, fmap;
  int kernel_size, dilation;            /* CONV_LIKE */
  int gather;               /* AXIAL_ROW / AXIAL_COL, bf16, training shapes only: gathered axial tiling, see below */
  int kv_rows;              /* forward only: rows allocated per (batch, head) in k and v (0 = n_k).  > n_k: an in-place KV cache --
                               k, v are [batch, heads, kv_rows, 64] buffers of which the first n_k rows are valid (attention.py:71-76
                               grows the cache with torch.cat instead); the rows behind them must hold finite values (zero-fill
                               the buffers once) */
  const uint8_t* key_mask;  /* optional [batch, n_k] 1 = keep (attention.py:80-83) */
  const uint8_t* static_mask; int64_t static_ld;   /* STATIC: [n, static_ld] 1 = allowed */
  const void* q; const void* k; const void* v;
  void* out;
  float* lse;
} db200_attn_fwd_params;
int dalle_b200_attn_fwd(const db200_attn_fwd_params* p, void* stream);

/* backward: d_out [batch, n, heads*64] (dtype) -> dqkv [batch*n, 3*heads*64] (dtype) = gradient w.r.t. the
 * to_qkv output, i.e. with the inverse rotary rotation and the q-scale folded in (attention.py:63-69 adjoint).
 * delta [batch, heads, n] fp32 is workspace.  Training only (n_q == n_k). */
typedef struct {
  db200_attn_fwd_params f;  /* same geometry / q,k,v / out / lse as the forward call */
  const void* d_out;
  const float* cos_t; const float* sin_t; float q_scale;  /* as in EPI_QKV; NULL tables = no rotary */
  float* delta;
  void* dqkv;
} db200_attn_bwd_params;
int dalle_b200_attn_bwd(const db200_attn_bwd_params* p, void* stream);

/* ---------------------------------------------------------------------------------------------
 * LayerScale / residual backward glue (transformer.py:88 adjoint + bias grad of the last Linear):
 *   dy[m,c]   = sign * scale[c] * d_out[m,c]          (dtype)  -> A operand of dgrad / wgrad
 *   dscale[c] += sum_m sign * d_out[m,c] * y[m,c]
 *   dbias[c]  += sum_m dy[m,c]
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  int rows, d;
  int dtype;
  float sign;
  const float* d_out;
  const void* y;            /* [rows,d] (dtype) saved by EPI_RESID; may be NULL when scale is NULL */
  const float* scale;       /* NULL = 1 */
  void* dy;
  float* dscale;            /* optional, += */
  float* dbias;             /* optional, += */
} db200_scale_bwd_params;
int dalle_b200_scale_bwd(const db200_scale_bwd_params* p, void* stream);

/* column sums: out[c] += sum_m x[m,c]  (bias gradient of net.0, transformer.py:114) */
int dalle_b200_colsum(const void* x, int dtype, int rows, int cols, float* out, void* stream);

/* Head split + rotary(q,k,v) + q scale as a streaming pass over the plain to_qkv output (the same math as EPI_QKV,
 * attention.py:63-69): qkv [rows, 3*heads*dim_head] -> q,k,v [rows/seq_n, heads, n_alloc, dim_head] (dtype).
 * n_alloc >= seq_n rows are laid out per (batch, head) (0 = seq_n); rows seq_n .. n_alloc-1 are written as zeros (the zero
 * token the reference's axial attention pads with, attention.py:255-258). */
int dalle_b200_qkv_rotary(const void* qkv, void* q, void* k, void* v, const float* cos_t, const float* sin_t, int dtype, int rows, int seq_n,
                          int heads, int dim_head, int pos_offset, float q_scale, int n_alloc, void* stream);

/* GEGLU adjoint as a streaming pass: dh [rows, hidden], u = [a|g] [rows, 2*hidden] -> du [rows, 2*hidden] (dtype);
 * dbias [2*hidden] fp32 (optional, +=) receives the column sums of du = gradient of net.0.bias (transformer.py:106-115) */
int dalle_b200_geglu_bwd(const void* dh, const void* u, void* du, float* dbias, int dtype, int rows, int hidden, void* stream);

/* Cross-entropy over the rows of logits [rows, vocab] (dtype) with int64 labels (F.cross_entropy, dalle_pytorch.py:667-668):
 * fwd: row_lse[r] = logsumexp(logits[r,:]);  *loss_acc += coef * sum_r (row_lse[r] - logits[r, labels[r]])   (coef = weight/rows)
 * bwd: logits[r,j] <- (*upstream) * coef * (exp(logits[r,j] - row_lse[r]) - [j == labels[r]])   IN PLACE (becomes d logits) */
int dalle_b200_ce_fwd(const void* logits, int dtype, int rows, int vocab, const int64_t* labels, float coef, float* row_lse, float* loss_acc,
                      void* stream);
int dalle_b200_ce_bwd(void* logits, int dtype, int rows, int vocab, const int64_t* labels, float coef, const float* row_lse, const float* upstream,
                      void* stream);

/* fp32 GEMMs on the bf16 tensor cores ("bf16x6" parity mode): split an fp32 matrix into three bf16 pieces x0 + x1 + x2 (24
 * mantissa bits) and lay the pieces out six times along the GEMM's K axis in the order operand A (operand = 0:
 * a0 a0 a1 a1 a0 a2) or operand B (operand = 1: b0 b1 b0 b1 b2 b0) needs, so that ONE dalle_b200_gemm call over K' = 6K with bf16
 * operands and an fp32 STORE result equals the fp32 product up to relative terms of 2^-24.
 *   concat_rows = 0: src [rows, cols] fp32 -> dst [rows, 6*cols] bf16  (K-major operand: K is the contiguous axis)
 *   concat_rows = 1: src [rows, cols] fp32 -> dst [6*rows, cols] bf16  (MN-major operand: K is the row index) */
int dalle_b200_split_bf16x3(const float* src, void* dst, int64_t rows, int cols, int concat_rows, int operand, void* stream);
/* out[r,c] = resid[r,c] + sign * scale[c] * y[r,c]   (resid / scale optional) -- the LayerScale + residual step of
 * EPI_RESID as a streaming pass (transformer.py:88, reversible.py:139-140), used by the bf16x6 parity mode and when dropout sits
 * between the projection and the LayerScale; y is `dtype`, everything else fp32 */
int dalle_b200_resid_scale(const void* y, int dtype, const float* resid, const float* scale, float sign, float* out, int64_t rows, int d, void* stream);
/* Decoding (generate_images, dalle_pytorch.py:533-539): out[r] = argmax_i(logits[r,i] / temperature + g[r,i]) over the k largest
 * logits of row r -- top_k(logits, thres) with k = max(int((1 - thres) * vocab), 1) followed by gumbel_sample, in one launch per
 * step.  g = -log(-log(u)) with u from Philox4x32-10(seed, offset + (r*vocab + i) / 4), or read from `gumbel` [rows, vocab] fp32 when
 * that pointer is not NULL (tests).  logits: [rows, ld] (dtype), out: int64 [rows]. */
int dalle_b200_sample_topk_gumbel(const void* logits, int dtype, int rows, int vocab, int64_t ld, int k, float temperature, const float* gumbel,
                                  uint64_t seed, uint64_t offset, int64_t* out, void* stream);
/* Classifier-free guidance (generate_images(cond_scale = s)): the same sampling for the guided logits null + (cond - null) * s of
 * rows [rows, vocab], formed element by element from cond [rows, ld] and null_logits [rows, ld] (dtype) and never written.  Each of
 * the three operations is rounded separately (fp32, then to dtype) as torch rounds `null + (cond - null) * s`, so the result -- and
 * with the same (seed, offset) the token -- equals dalle_b200_sample_topk_gumbel on torch's guided logits. */
int dalle_b200_sample_guided_topk_gumbel(const void* cond, const void* null_logits, int dtype, int rows, int vocab, int64_t ld, float cond_scale, int k,
                                         float temperature, const float* gumbel, uint64_t seed, uint64_t offset, int64_t* out, void* stream);
/* Graph-replayed decoding (dalle_pytorch_b200/decode.py): one new token per sequence, its POSITION read from device memory (`pos`,
 * one int64) so that one captured launch sequence serves every token.
 * decode_shift: PreShiftToken's cache branch (reference transformer.py:155-170) for the token at position *pos.  h [batch, d] fp32 =
 * the token after PreNorm; ring_top [fmap, batch, d/4], ring_left [fmap, batch, d/2 - d/4] fp32 = the first-half channels of the
 * last `fmap` image tokens, slot = (position - text_len) mod fmap.  y [batch, d] (out_dtype) = [ring_top[slot] | ring_left[slot-1]
 * (zeros when slot == 0) | h[d/2:]]; the token's own first half replaces ring slot `slot`. */
int dalle_b200_decode_shift(const float* h, void* y, int out_dtype, int batch, int d, float* ring_top, float* ring_left, const int64_t* pos,
                            int text_len, int fmap, void* stream);
/* decode_kv_append: k_new / v_new [batch_heads, dim_head] -> row *pos of the in-place caches k_cache / v_cache
 * [batch_heads, kv_rows, dim_head] (reference attention.py:71-76 re-allocates the cache with torch.cat instead). */
int dalle_b200_decode_kv_append(const void* k_new, const void* v_new, void* k_cache, void* v_cache, int dtype, int batch_heads, int dim_head,
                                int kv_rows, const int64_t* pos, void* stream);

/* Dropout with a counter-based generator (attention.py:53-56, transformer.py:117): y[i] = keep(i) ? x[i] / (1 - p) : 0 where
 * keep(i) = word (i & 3) of Philox4x32-10(key = seed, counter = offset + i / 4) <= (1 - p) * 2^32.  In place allowed (y == x).
 * The mask is a pure function of (seed, offset, i): pass the same pair to the backward pass (on the gradient) and to the
 * reversible executor's recomputation -- the library's form of Deterministic.record_rng / set_rng (reversible.py:20-50). */
int dalle_b200_dropout(const void* x, void* y, int dtype, int64_t count, float p, uint64_t seed, uint64_t offset, void* stream);
/* h[r,j] = u[r,j] * gelu_erf(u[r,hidden+j])   (fp32; transformer.py:106-109) -- the GEGLU step of EPI_GEGLU as a streaming pass */
int dalle_b200_geglu_fwd(const float* u, float* h, int64_t rows, int hidden, void* stream);

/* mc_dst[i] += scale * src[i] on EVERY GPU's copy of a symmetric buffer (multimem.red through the NVLink multicast address
 * `mc_dst`, 16-byte aligned): how gradients that are not produced by a weight-gradient GEMM join the data-parallel sum. */
int dalle_b200_mc_add(const float* src, void* mc_dst, int64_t count, float scale, void* stream);

/* fp32 -> bf16 cast of `count` elements (weights are kept in fp32 and cast once per step) */
int dalle_b200_cast_bf16(const float* src, void* dst, int64_t count, void* stream);

/* y = a + alpha*b over fp32 (reversible stream arithmetic, reversible.py:83,86,96,99) */
int dalle_b200_axpby(const float* a, const float* b, float alpha, float* y, int64_t count, void* stream);

/* Token embedding written straight into the [batch, n, d] fp32 token stream (dalle_pytorch.py:616-630: text_emb / image_emb
 * lookups + torch.cat): out[b, seg_off + l, :] = weight[ids[b, l], :] for l < seg_len.  ids are int64, 0 <= id < vocab.
 * The backward adds d_out[b, seg_off + l, :] into dweight[ids[b, l], :] with fp32 atomics (dweight zero-initialised or
 * carrying a previous accumulation), replacing nn.Embedding's sort-based gradient. */
int dalle_b200_embed_fwd(const int64_t* ids, const float* weight, float* out, int batch, int seg_len, int n, int seg_off, int d, int vocab,
                         void* stream);
int dalle_b200_embed_bwd(const int64_t* ids, const float* d_out, float* dweight, int batch, int seg_len, int n, int seg_off, int d, int vocab,
                         void* stream);

/* Optimizer step of the reference trainer (train_dalle.py:617-619: clip_grad_norm_(params, 0.5); Adam.step()) over FLAT fp32
 * buffers, two launches for the whole model:
 *   dalle_b200_sumsq   : *out += sum(x[i]^2)                      (out: fp32 device scalar, caller zeroes it)
 *   dalle_b200_adam    : coef = max_norm > 0 ? min(1, max_norm / (sqrt(*gnorm_sq) + 1e-6)) : 1     (clip_grad_norm_)
 *                        g = coef * grad (+ weight_decay * p);  m = b1 m + (1-b1) g;  v = b2 v + (1-b2) g^2;
 *                        p -= (lr / (1 - b1^step)) * m / (sqrt(v) / sqrt(1 - b2^step) + eps)        (torch.optim.Adam)
 * The clip coefficient is read on the device, so the step needs no host synchronisation. */
int dalle_b200_sumsq(const float* x, int64_t count, float* out, void* stream);
typedef struct {
  float* p; const float* g; float* m; float* v;      /* [count] fp32 each */
  int64_t count;
  float lr, beta1, beta2, eps, weight_decay;
  int step;                                          /* 1-based */
  float max_norm;                                    /* <= 0: no clipping */
  const float* gnorm_sq;                             /* device scalar from dalle_b200_sumsq (may be NULL when max_norm <= 0) */
} db200_adam_params;
int dalle_b200_adam(const db200_adam_params* p, void* stream);

/* Debug export, NOT part of the contract (no reference counterpart): clock64() timeline of one dK/dV attention CTA recorded when
 * DALLE_B200_ATTN_WAIT has bit 2 set; used by tools/attn_timeline.py. */
int dalle_b200_debug_attn_timeline(long long* out, int count);

#ifdef __cplusplus
}
#endif
#endif /* DALLE_B200_H */
