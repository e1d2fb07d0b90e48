// C ABI of libdalle_b200.so (include/dalle_b200.h): argument validation and dispatch to the kernels.
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "common.cuh"

namespace db200 {
bool pdl_enabled() {
  static const bool on = [] { const char* v = std::getenv("DALLE_B200_PDL"); return !(v && v[0] == '0'); }();
  return on;
}

std::string& last_error_slot() {
  static thread_local std::string s;
  return s;
}

int set_error(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  last_error_slot() = buf;
  return code;
}

int sm_count() {
  static std::atomic<int> cached[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

// kernels (other translation units)
int ln_shift_fwd_launch(const db200_ln_shift_fwd_params& P, cudaStream_t st);
int ln_shift_bwd_launch(const db200_ln_shift_bwd_params& P, cudaStream_t st);
int scale_bwd_launch(const db200_scale_bwd_params& P, cudaStream_t st);
int colsum_launch(const void* x, int dtype, int rows, int cols, float* out, cudaStream_t st);
int ce_fwd_launch(const void* logits, int dtype, int rows, int vocab, const long long* labels, float coef, float* row_lse, float* loss_acc, cudaStream_t st);
int ce_bwd_launch(void* logits, int dtype, int rows, int vocab, const long long* labels, float coef, const float* row_lse, const float* upstream, cudaStream_t st);
int qkv_rotary_launch(const void* qkv, void* q, void* k, void* v, const float* cos_t, const float* sin_t, int dtype, int rows, int seq_n, int heads,
                      int dh, int pos_offset, float q_scale, int n_alloc, cudaStream_t st);
int geglu_bwd_launch(const void* dh, const void* u, void* du, float* dbias, int dtype, int rows, int hidden, cudaStream_t st);
int cast_bf16_launch(const float* src, void* dst, int64_t count, cudaStream_t st);
int split_bf16x3_launch(const float* src, void* dst, int64_t rows, int cols, int concat_rows, int pat, cudaStream_t st);
int resid_scale_launch(const void* y, int dtype, const float* resid, const float* scale, float sign, float* out, int64_t rows, int d, cudaStream_t st);
int mc_add_launch(const float* src, void* mc_dst, int64_t count, float scale, cudaStream_t st);
int sample_topk_gumbel_launch(const void* logits, int dtype, int rows, int vocab, long long ld, int k, float temperature, const float* gumbel,
                              unsigned long long seed, unsigned long long offset, long long* out, cudaStream_t st);
int sample_guided_topk_gumbel_launch(const void* cond, const void* null_logits, int dtype, int rows, int vocab, long long ld, float cond_scale, int k,
                                     float temperature, const float* gumbel, unsigned long long seed, unsigned long long offset, long long* out,
                                     cudaStream_t st);
int dropout_launch(const void* x, void* y, int dtype, int64_t count, float p, unsigned long long seed, unsigned long long offset, cudaStream_t st);
int geglu_fwd_launch(const float* u, float* h, int64_t rows, int hidden, cudaStream_t st);
int axpby_launch(const float* a, const float* b, float alpha, float* y, int64_t count, cudaStream_t st);
int sumsq_launch(const float* x, int64_t count, float* out, cudaStream_t st);
int adam_launch(const db200_adam_params& P, cudaStream_t st);
int embed_launch(bool bwd, const long long* ids, const float* a, float* o, int batch, int seg_len, int n, int seg_off, int d, int vocab, cudaStream_t st);
int gemm_simt_launch(const db200_gemm_params& p, cudaStream_t st);
bool gemm_tcgen05_supported(const db200_gemm_params& p, const char** why);
int gemm_tcgen05_launch(const db200_gemm_params& p, cudaStream_t st);
bool gemm_smallm_supported(const db200_gemm_params& p, const char** why);
int gemm_smallm_launch(const db200_gemm_params& p, cudaStream_t st);
int attn_fwd_simt_launch(const db200_attn_fwd_params& p, cudaStream_t st);
int attn_bwd_simt_launch(const db200_attn_bwd_params& p, cudaStream_t st);
bool attn_mma_supported(const db200_attn_fwd_params& p);
int attn_fwd_mma_launch(const db200_attn_fwd_params& p, cudaStream_t st);
int attn_bwd_mma_launch(const db200_attn_bwd_params& p, cudaStream_t st);
bool attn_tc_supported(const db200_attn_fwd_params& p);
bool attn_gather_ok(const db200_attn_fwd_params& p, const char** why);
int attn_fwd_tc_launch(const db200_attn_fwd_params& p, cudaStream_t st);
int attn_bwd_tc_launch(const db200_attn_bwd_params& p, cudaStream_t st);
int attn_debug_timeline(long long* out, int count);
bool attn_decode_supported(const db200_attn_fwd_params& p);
int attn_decode_launch(const db200_attn_fwd_params& p, cudaStream_t st);
int decode_shift_launch(const float* h, void* y, int out_dtype, int batch, int d, float* ring_top, float* ring_left, const long long* pos,
                        int text_len, int fmap, cudaStream_t st);
int decode_kv_append_launch(const void* k_new, const void* v_new, void* k_cache, void* v_cache, int dtype, int bh, int dh, int kv_rows,
                            const long long* pos, cudaStream_t st);

static bool dtype_ok(int d) { return d == DB200_F32 || d == DB200_BF16; }
static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// DALLE_B200_GEMM=simt|tcgen05 and DALLE_B200_ATTN=simt|mma override the AUTO choice (debugging / A-B timing)
static int env_choice(const char* name, const char* a, const char* b) {
  const char* v = getenv(name);
  if (!v) return 0;
  if (!strcmp(v, a)) return 1;
  if (!strcmp(v, b)) return 2;
  return 0;
}

}  // namespace db200

using namespace db200;

extern "C" {

int dalle_b200_version(void) { return DALLE_B200_VERSION; }
// debug probe (not part of the documented ABI): clock64() timeline of one dK/dV CTA, see attn_tc.cu
int dalle_b200_debug_attn_timeline(long long* out, int count) { return db200::attn_debug_timeline(out, count); }

const char* dalle_b200_last_error(void) { return last_error_slot().c_str(); }

int dalle_b200_device_ok(int dev) {
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) return 0;
  return prop.major == 10 ? 1 : 0;
}

int dalle_b200_abi_sizes(int* out, int capacity) {
  const int sizes[7] = {(int)sizeof(db200_ln_shift_fwd_params), (int)sizeof(db200_ln_shift_bwd_params), (int)sizeof(db200_gemm_params),
                        (int)sizeof(db200_attn_fwd_params),     (int)sizeof(db200_attn_bwd_params),     (int)sizeof(db200_scale_bwd_params),
                        (int)sizeof(db200_adam_params)};
  for (int i = 0; i < 7 && i < capacity; ++i) out[i] = sizes[i];
  return 7;
}

int dalle_b200_ln_shift_fwd(const db200_ln_shift_fwd_params* p, void* stream) {
  DB200_CHECK_ARG(p != nullptr, "ln_shift_fwd: null params");
  DB200_CHECK_ARG(p->batch >= 0 && p->n >= 0 && p->d > 0, "ln_shift_fwd: bad shape b=%d n=%d d=%d", p->batch, p->n, p->d);
  DB200_CHECK_ARG(dtype_ok(p->out_dtype), "ln_shift_fwd: bad dtype %d", p->out_dtype);
  DB200_CHECK_ARG(p->d % (p->do_shift ? 16 : 4) == 0, "ln_shift_fwd: d=%d must be a multiple of %d", p->d, p->do_shift ? 16 : 4);
  DB200_CHECK_ARG(p->x && p->out, "ln_shift_fwd: null tensor");
  DB200_CHECK_ARG(aligned16(p->x) && aligned16(p->out), "ln_shift_fwd: tensors must be 16-byte aligned");
  if (p->do_ln) DB200_CHECK_ARG(p->gamma && p->beta && p->mean && p->rstd, "ln_shift_fwd: LayerNorm needs gamma/beta/mean/rstd");
  if (p->do_shift) {
    DB200_CHECK_ARG(p->fmap > 0 && p->text_len > 0, "ln_shift_fwd: shift needs text_len/fmap");
    DB200_CHECK_ARG(p->n >= p->text_len, "ln_shift_fwd: n=%d < text_len=%d is the no-shift case (transformer.py:160)", p->n, p->text_len);
    DB200_CHECK_ARG(p->n <= p->text_len + p->fmap * p->fmap, "ln_shift_fwd: n=%d exceeds text_len + fmap^2", p->n);
  }
  return ln_shift_fwd_launch(*p, (cudaStream_t)stream);
}

int dalle_b200_ln_shift_bwd(const db200_ln_shift_bwd_params* p, void* stream) {
  DB200_CHECK_ARG(p != nullptr, "ln_shift_bwd: null params");
  DB200_CHECK_ARG(p->batch >= 0 && p->n >= 0 && p->d > 0, "ln_shift_bwd: bad shape");
  DB200_CHECK_ARG(dtype_ok(p->dout_dtype), "ln_shift_bwd: bad dtype %d", p->dout_dtype);
  DB200_CHECK_ARG(p->d % (p->do_shift ? 16 : 4) == 0, "ln_shift_bwd: d=%d alignment", p->d);
  DB200_CHECK_ARG(p->d_out && p->dx, "ln_shift_bwd: null tensor");
  if (p->do_ln) DB200_CHECK_ARG(p->x && p->mean && p->rstd && p->gamma && p->dgamma && p->dbeta, "ln_shift_bwd: LayerNorm needs x/mean/rstd/gamma/dgamma/dbeta");
  if (p->do_shift) DB200_CHECK_ARG(p->fmap > 0 && p->n >= p->text_len && p->n <= p->text_len + p->fmap * p->fmap, "ln_shift_bwd: bad shift geometry");
  if (p->up_dy) {
    DB200_CHECK_ARG(p->d == 1024, "ln_shift_bwd: the fused upstream LayerScale adjoint needs d = 1024 (got %d)", p->d);
    DB200_CHECK_ARG(aligned16(p->up_dy) && aligned16(p->up_y) && aligned16(p->d_out) && aligned16(p->x) && aligned16(p->dres),
                    "ln_shift_bwd: fused path needs 16-byte aligned tensors");
    DB200_CHECK_ARG(p->up_dscale == nullptr || p->up_y != nullptr, "ln_shift_bwd: up_dscale needs up_y");
  }
  return ln_shift_bwd_launch(*p, (cudaStream_t)stream);
}

int dalle_b200_gemm(const db200_gemm_params* p, void* stream) {
  DB200_CHECK_ARG(p != nullptr, "gemm: null params");
  DB200_CHECK_ARG(p->M >= 0 && p->N > 0 && p->K > 0, "gemm: bad shape M=%d N=%d K=%d", p->M, p->N, p->K);
  DB200_CHECK_ARG(dtype_ok(p->dtype), "gemm: bad dtype %d", p->dtype);
  DB200_CHECK_ARG(p->A && p->B, "gemm: null operand");
  DB200_CHECK_ARG((p->N & 1) == 0, "gemm: N=%d must be even (epilogues work on column pairs)", p->N);
  switch (p->epilogue) {
    case DB200_EPI_STORE:
      DB200_CHECK_ARG(p->C && dtype_ok(p->c_dtype) && (p->ldc & 1) == 0, "gemm/STORE: bad C");
      if (p->C_multicast)
        DB200_CHECK_ARG(p->c_dtype == DB200_F32 && p->bias == nullptr && aligned16(p->C_multicast) && (p->ldc & 3) == 0 && p->backend != DB200_GEMM_SIMT,
                        "gemm/STORE: the multicast reduction needs an fp32 result, no bias, 16-byte aligned rows and the tcgen05 kernel");
      break;
    case DB200_EPI_QKV:
      DB200_CHECK_ARG(p->q && p->k && p->v, "gemm/QKV: null q/k/v");
      DB200_CHECK_ARG(p->heads > 0 && p->dim_head > 0 && (p->dim_head & 1) == 0 && p->N == 3 * p->heads * p->dim_head,
                      "gemm/QKV: N=%d != 3*heads*dim_head (%d*%d)", p->N, p->heads, p->dim_head);
      DB200_CHECK_ARG(p->seq_n > 0 && p->M % p->seq_n == 0, "gemm/QKV: M=%d not a multiple of seq_n=%d", p->M, p->seq_n);
      DB200_CHECK_ARG((p->cos_t == nullptr) == (p->sin_t == nullptr), "gemm/QKV: cos/sin tables must come together");
      break;
    case DB200_EPI_RESID:
      DB200_CHECK_ARG(p->out != nullptr, "gemm/RESID: null out");
      break;
    case DB200_EPI_GEGLU:
      DB200_CHECK_ARG(p->h_out && p->hidden > 0 && p->N == 2 * p->hidden && (p->hidden & 1) == 0, "gemm/GEGLU: N must equal 2*hidden");
      break;
    case DB200_EPI_GEGLU_BWD:
      DB200_CHECK_ARG(p->u_in && p->du_out && p->hidden == p->N, "gemm/GEGLU_BWD: N must equal hidden");
      break;
    default:
      return set_error(DB200_ERR_BAD_ARG, "gemm: unknown epilogue %d", p->epilogue);
  }
  if (p->M == 0) return DB200_OK;
  int backend = p->backend;
  if (backend == DB200_GEMM_SMALLM) {
    const char* why = "";
    if (!gemm_smallm_supported(*p, &why)) return set_error(DB200_ERR_UNSUPPORTED, "gemm: the small-M kernel cannot run this problem: %s", why);
    return gemm_smallm_launch(*p, (cudaStream_t)stream);
  }
  if (backend == DB200_GEMM_AUTO) {
    const int env = env_choice("DALLE_B200_GEMM", "simt", "tcgen05");
    if (env == 1) backend = DB200_GEMM_SIMT;
    else {
      const char* why = nullptr;
      backend = gemm_tcgen05_supported(*p, &why) ? DB200_GEMM_TCGEN05 : DB200_GEMM_SIMT;
    }
  }
  if (p->C_multicast && backend != DB200_GEMM_TCGEN05)
    return set_error(DB200_ERR_UNSUPPORTED, "gemm/STORE: the multicast reduction is implemented by the tcgen05 kernel only (shape / alignment did not qualify)");
  if (backend == DB200_GEMM_TCGEN05) {
    const char* why = "";
    if (!gemm_tcgen05_supported(*p, &why)) return set_error(DB200_ERR_UNSUPPORTED, "gemm: tcgen05 backend cannot run this problem: %s", why);
    return gemm_tcgen05_launch(*p, (cudaStream_t)stream);
  }
  return gemm_simt_launch(*p, (cudaStream_t)stream);
}

int dalle_b200_gemm_select(const db200_gemm_params* p) {
  if (!p) return DB200_GEMM_SIMT;
  if (p->backend != DB200_GEMM_AUTO) return p->backend;
  if (env_choice("DALLE_B200_GEMM", "simt", "tcgen05") == 1) return DB200_GEMM_SIMT;
  const char* why = nullptr;
  return gemm_tcgen05_supported(*p, &why) ? DB200_GEMM_TCGEN05 : DB200_GEMM_SIMT;
}

// 0 = CUDA-core fp32 arithmetic, 1 = mma.sync bf16, 2 = tcgen05 bf16
static int attn_backend(const db200_attn_fwd_params& f) {
  const char* v = getenv("DALLE_B200_ATTN");
  int want = 2;                                   // tcgen05 kernels (attn_tc.cu) whenever the problem qualifies
  if (f.gather) return 2;                         // validated by check_attn
  if (v) want = !strcmp(v, "simt") ? 0 : !strcmp(v, "tc") ? 2 : 1;
  if (want == 2 && !attn_tc_supported(f)) want = 1;
  if (want == 1 && !attn_mma_supported(f)) want = 0;
  return want;
}

static int check_attn(const db200_attn_fwd_params& f, const char* who) {
  DB200_CHECK_ARG(f.batch >= 0 && f.heads > 0 && f.n_q >= 0 && f.n_k >= f.n_q, "%s: bad shape", who);
  if (f.dim_head != 64) return set_error(DB200_ERR_UNSUPPORTED, "%s: dim_head=%d, kernels are specialised for 64", who, f.dim_head);
  DB200_CHECK_ARG(dtype_ok(f.dtype), "%s: bad dtype", who);
  DB200_CHECK_ARG(f.q && f.k && f.v && f.out && f.lse, "%s: null tensor", who);
  DB200_CHECK_ARG(f.pattern >= DB200_ATTN_FULL && f.pattern <= DB200_ATTN_STATIC, "%s: bad pattern %d", who, f.pattern);
  if (f.pattern == DB200_ATTN_STATIC) DB200_CHECK_ARG(f.static_mask && f.static_ld >= f.n_k, "%s: STATIC needs static_mask", who);
  if (f.pattern == DB200_ATTN_AXIAL_ROW || f.pattern == DB200_ATTN_AXIAL_COL || f.pattern == DB200_ATTN_CONV_LIKE)
    DB200_CHECK_ARG(f.fmap > 0 && f.text_len > 0, "%s: sparse pattern needs text_len / fmap", who);
  if (f.pattern == DB200_ATTN_CONV_LIKE) DB200_CHECK_ARG(f.kernel_size > 0 && (f.kernel_size & 1) && f.dilation > 0, "%s: conv_like kernel_size must be odd", who);
  DB200_CHECK_ARG(f.kv_rows == 0 || (f.kv_rows >= f.n_k && !f.gather), "%s: kv_rows must be >= n_k (and is not combined with gather)", who);
  if (f.gather) {      // the caller has laid q/k/v/lse out for the gathered kernels: there is no other backend to fall back to
    const char* why = nullptr;
    if (!attn_gather_ok(f, &why)) return set_error(DB200_ERR_UNSUPPORTED, "%s: %s", who, why);
    if (!attn_tc_supported(f)) return set_error(DB200_ERR_UNSUPPORTED, "%s: gathered axial attention needs the tcgen05 path (sm_100, 16-byte aligned tensors)", who);
  }
  return DB200_OK;
}

int dalle_b200_attn_fwd(const db200_attn_fwd_params* p, void* stream) {
  DB200_CHECK_ARG(p != nullptr, "attn_fwd: null params");
  const int rc = check_attn(*p, "attn_fwd");
  if (rc) return rc;
  if (p->batch == 0 || p->n_q == 0) return DB200_OK;
  // one query per head (KV-cache decoding, bf16): the streaming kernel of decode.cu instead of a 128-query tile
  if (attn_decode_supported(*p)) return attn_decode_launch(*p, (cudaStream_t)stream);
  // DALLE_B200_ATTN = simt | mma | tc   (default: see attn_default_backend)
  const int be = attn_backend(*p);
  if (be == 2) return attn_fwd_tc_launch(*p, (cudaStream_t)stream);
  if (be == 1) return attn_fwd_mma_launch(*p, (cudaStream_t)stream);
  return attn_fwd_simt_launch(*p, (cudaStream_t)stream);
}

int dalle_b200_attn_bwd(const db200_attn_bwd_params* p, void* stream) {
  DB200_CHECK_ARG(p != nullptr, "attn_bwd: null params");
  const int rc = check_attn(p->f, "attn_bwd");
  if (rc) return rc;
  DB200_CHECK_ARG(p->f.kv_rows == 0 || p->f.kv_rows == p->f.n_k, "attn_bwd: kv_rows (in-place KV cache) is a forward-only layout");
  DB200_CHECK_ARG(p->f.n_q == p->f.n_k, "attn_bwd: training only (n_q == n_k)");
  DB200_CHECK_ARG(p->d_out && p->delta && p->dqkv, "attn_bwd: null tensor");
  DB200_CHECK_ARG((p->cos_t == nullptr) == (p->sin_t == nullptr), "attn_bwd: cos/sin tables must come together");
  if (p->f.batch == 0 || p->f.n_q == 0) return DB200_OK;
  const int be = attn_backend(p->f);
  if (be == 2) return attn_bwd_tc_launch(*p, (cudaStream_t)stream);
  if (be == 1) return attn_bwd_mma_launch(*p, (cudaStream_t)stream);
  return attn_bwd_simt_launch(*p, (cudaStream_t)stream);
}

int dalle_b200_scale_bwd(const db200_scale_bwd_params* p, void* stream) {
  DB200_CHECK_ARG(p != nullptr, "scale_bwd: null params");
  DB200_CHECK_ARG(p->rows >= 0 && p->d > 0 && (p->d & 1) == 0, "scale_bwd: bad shape");
  DB200_CHECK_ARG(dtype_ok(p->dtype) && p->d_out && p->dy, "scale_bwd: bad args");
  return scale_bwd_launch(*p, (cudaStream_t)stream);
}

int dalle_b200_colsum(const void* x, int dtype, int rows, int cols, float* out, void* stream) {
  DB200_CHECK_ARG(x && out && rows >= 0 && cols > 0 && (cols & 1) == 0 && dtype_ok(dtype), "colsum: bad args");
  return colsum_launch(x, dtype, rows, cols, out, (cudaStream_t)stream);
}

int dalle_b200_geglu_bwd(const void* dh, const void* u, void* du, float* dbias, int dtype, int rows, int hidden, void* stream) {
  DB200_CHECK_ARG(dh && u && du && rows >= 0 && hidden > 0 && (hidden & 7) == 0 && dtype_ok(dtype), "geglu_bwd: bad args (hidden must be a multiple of 8)");
  DB200_CHECK_ARG(aligned16(dh) && aligned16(u) && aligned16(du), "geglu_bwd: tensors must be 16-byte aligned");
  return geglu_bwd_launch(dh, u, du, dbias, dtype, rows, hidden, (cudaStream_t)stream);
}

int dalle_b200_qkv_rotary(const void* qkv, void* q, void* k, void* v, const float* cos_t, const float* sin_t, int dtype, int rows, int seq_n,
                          int heads, int dim_head, int pos_offset, float q_scale, int n_alloc, void* stream) {
  if (n_alloc == 0) n_alloc = seq_n;
  DB200_CHECK_ARG(n_alloc >= seq_n, "qkv_rotary: n_alloc must be >= seq_n");
  DB200_CHECK_ARG(qkv && q && k && v && dtype_ok(dtype) && rows >= 0 && seq_n > 0 && heads > 0 && dim_head > 0 && (dim_head & 7) == 0 &&
                      rows % seq_n == 0,
                  "qkv_rotary: bad args (dim_head must be a multiple of 8, rows a multiple of seq_n)");
  DB200_CHECK_ARG((cos_t == nullptr) == (sin_t == nullptr), "qkv_rotary: cos/sin tables must come together");
  DB200_CHECK_ARG(aligned16(qkv) && aligned16(q) && aligned16(k) && aligned16(v) && (!cos_t || (aligned16(cos_t) && aligned16(sin_t))),
                  "qkv_rotary: tensors must be 16-byte aligned");
  return qkv_rotary_launch(qkv, q, k, v, cos_t, sin_t, dtype, rows, seq_n, heads, dim_head, pos_offset, q_scale, n_alloc, (cudaStream_t)stream);
}

int dalle_b200_split_bf16x3(const float* src, void* dst, int64_t rows, int cols, int concat_rows, int operand, void* stream) {
  DB200_CHECK_ARG(src && dst && rows >= 0 && cols > 0 && (cols & 1) == 0 && (operand == 0 || operand == 1), "split_bf16x3: bad args (cols must be even)");
  DB200_CHECK_ARG(aligned16(src) && aligned16(dst), "split_bf16x3: tensors must be 16-byte aligned");
  // K-block -> piece: products (a0 b0) (a0 b1) (a1 b0) (a1 b1) (a0 b2) (a2 b0)
  // (nibble blk = piece held by K block blk)   A: a0 a0 a1 a1 a0 a2      B: b0 b1 b0 b1 b2 b0
  const int pat = operand == 0 ? 0x201100 : 0x021010;
  return split_bf16x3_launch(src, dst, rows, cols, concat_rows != 0, pat, (cudaStream_t)stream);
}

int dalle_b200_resid_scale(const void* y, int dtype, const float* resid, const float* scale, float sign, float* out, int64_t rows, int d, void* stream) {
  DB200_CHECK_ARG(y && out && rows >= 0 && d > 0 && (d & 1) == 0 && dtype_ok(dtype), "resid_scale: bad args (d must be even)");
  return resid_scale_launch(y, dtype, resid, scale, sign, out, rows, d, (cudaStream_t)stream);
}

int dalle_b200_mc_add(const float* src, void* mc_dst, int64_t count, float scale, void* stream) {
  DB200_CHECK_ARG(src && mc_dst && count >= 0 && aligned16(src) && aligned16(mc_dst), "mc_add: bad args (16-byte aligned fp32 buffers)");
  return mc_add_launch(src, mc_dst, count, scale, (cudaStream_t)stream);
}

int dalle_b200_sample_topk_gumbel(const void* logits, int dtype, int rows, int vocab, int64_t ld, int k, float temperature, const float* gumbel,
                                  uint64_t seed, uint64_t offset, int64_t* out, void* stream) {
  DB200_CHECK_ARG(logits && out && rows >= 0 && vocab > 0 && ld >= vocab && dtype_ok(dtype), "sample_topk_gumbel: bad args");
  DB200_CHECK_ARG(k >= 1 && k <= vocab && temperature > 0.f, "sample_topk_gumbel: need 1 <= k <= vocab and temperature > 0");
  if ((size_t)vocab * 4 > 200 * 1024) return set_error(DB200_ERR_UNSUPPORTED, "sample_topk_gumbel: vocab=%d does not fit the shared-memory row buffer", vocab);
  return sample_topk_gumbel_launch(logits, dtype, rows, vocab, ld, k, temperature, gumbel, seed, offset, reinterpret_cast<long long*>(out), (cudaStream_t)stream);
}

int dalle_b200_sample_guided_topk_gumbel(const void* cond, const void* null_logits, int dtype, int rows, int vocab, int64_t ld, float cond_scale, int k,
                                         float temperature, const float* gumbel, uint64_t seed, uint64_t offset, int64_t* out, void* stream) {
  DB200_CHECK_ARG(cond && null_logits && out && rows >= 0 && vocab > 0 && ld >= vocab && dtype_ok(dtype), "sample_guided_topk_gumbel: bad args");
  DB200_CHECK_ARG(k >= 1 && k <= vocab && temperature > 0.f, "sample_guided_topk_gumbel: need 1 <= k <= vocab and temperature > 0");
  if ((size_t)vocab * 4 > 200 * 1024) return set_error(DB200_ERR_UNSUPPORTED, "sample_guided_topk_gumbel: vocab=%d does not fit the shared-memory row buffer", vocab);
  return sample_guided_topk_gumbel_launch(cond, null_logits, dtype, rows, vocab, ld, cond_scale, k, temperature, gumbel, seed, offset,
                                          reinterpret_cast<long long*>(out), (cudaStream_t)stream);
}

int dalle_b200_decode_shift(const float* h, void* y, int out_dtype, int batch, int d, float* ring_top, float* ring_left, const int64_t* pos,
                            int text_len, int fmap, void* stream) {
  DB200_CHECK_ARG(h && y && ring_top && ring_left && pos && dtype_ok(out_dtype), "decode_shift: null tensor / bad dtype");
  DB200_CHECK_ARG(batch >= 0 && d > 0 && (d & 3) == 0 && fmap > 0 && text_len >= 0, "decode_shift: bad shape (d must be a multiple of 4)");
  return decode_shift_launch(h, y, out_dtype, batch, d, ring_top, ring_left, reinterpret_cast<const long long*>(pos), text_len, fmap, (cudaStream_t)stream);
}

int dalle_b200_decode_kv_append(const void* k_new, const void* v_new, void* k_cache, void* v_cache, int dtype, int batch_heads, int dim_head,
                                int kv_rows, const int64_t* pos, void* stream) {
  DB200_CHECK_ARG(k_new && v_new && k_cache && v_cache && pos && dtype_ok(dtype), "decode_kv_append: null tensor / bad dtype");
  DB200_CHECK_ARG(batch_heads >= 0 && dim_head > 0 && kv_rows > 0, "decode_kv_append: bad shape");
  return decode_kv_append_launch(k_new, v_new, k_cache, v_cache, dtype, batch_heads, dim_head, kv_rows, reinterpret_cast<const long long*>(pos), (cudaStream_t)stream);
}

int dalle_b200_dropout(const void* x, void* y, int dtype, int64_t count, float p, uint64_t seed, uint64_t offset, void* stream) {
  DB200_CHECK_ARG(x && y && count >= 0 && dtype_ok(dtype) && p >= 0.f && p <= 1.f, "dropout: bad args (0 <= p <= 1)");
  return dropout_launch(x, y, dtype, count, p, seed, offset, (cudaStream_t)stream);
}

int dalle_b200_geglu_fwd(const float* u, float* h, int64_t rows, int hidden, void* stream) {
  DB200_CHECK_ARG(u && h && rows >= 0 && hidden > 0, "geglu_fwd: bad args");
  return geglu_fwd_launch(u, h, rows, hidden, (cudaStream_t)stream);
}

int dalle_b200_ce_fwd(const void* logits, int dtype, int rows, int vocab, const int64_t* labels, float coef, float* row_lse, float* loss_acc,
                      void* stream) {
  DB200_CHECK_ARG(logits && labels && row_lse && loss_acc && rows >= 0 && vocab > 0 && (vocab & 7) == 0 && dtype_ok(dtype),
                  "ce_fwd: bad args (vocab must be a multiple of 8)");
  DB200_CHECK_ARG(aligned16(logits), "ce_fwd: logits must be 16-byte aligned");
  return ce_fwd_launch(logits, dtype, rows, vocab, reinterpret_cast<const long long*>(labels), coef, row_lse, loss_acc, (cudaStream_t)stream);
}

int dalle_b200_ce_bwd(void* logits, int dtype, int rows, int vocab, const int64_t* labels, float coef, const float* row_lse, const float* upstream,
                      void* stream) {
  DB200_CHECK_ARG(logits && labels && row_lse && upstream && rows >= 0 && vocab > 0 && (vocab & 7) == 0 && dtype_ok(dtype), "ce_bwd: bad args");
  DB200_CHECK_ARG(aligned16(logits), "ce_bwd: logits must be 16-byte aligned");
  return ce_bwd_launch(logits, dtype, rows, vocab, reinterpret_cast<const long long*>(labels), coef, row_lse, upstream, (cudaStream_t)stream);
}

int dalle_b200_cast_bf16(const float* src, void* dst, int64_t count, void* stream) {
  DB200_CHECK_ARG(src && dst && count >= 0, "cast_bf16: bad args");
  DB200_CHECK_ARG(aligned16(src) && (reinterpret_cast<uintptr_t>(dst) & 7) == 0, "cast_bf16: alignment");
  return cast_bf16_launch(src, dst, count, (cudaStream_t)stream);
}

int dalle_b200_sumsq(const float* x, int64_t count, float* out, void* stream) {
  DB200_CHECK_ARG(x && out && count >= 0, "sumsq: bad args");
  DB200_CHECK_ARG(aligned16(x), "sumsq: x must be 16-byte aligned");
  return sumsq_launch(x, count, out, (cudaStream_t)stream);
}
int dalle_b200_adam(const db200_adam_params* p, void* stream) {
  DB200_CHECK_ARG(p != nullptr, "adam: null params");
  DB200_CHECK_ARG(p->p && p->g && p->m && p->v && p->count >= 0, "adam: null tensor / bad count");
  DB200_CHECK_ARG(aligned16(p->p) && aligned16(p->g) && aligned16(p->m) && aligned16(p->v), "adam: buffers must be 16-byte aligned");
  DB200_CHECK_ARG(p->step >= 1 && p->beta1 >= 0.f && p->beta1 < 1.f && p->beta2 >= 0.f && p->beta2 < 1.f && p->eps > 0.f, "adam: bad hyper-parameters");
  DB200_CHECK_ARG(p->max_norm <= 0.f || p->gnorm_sq != nullptr, "adam: clipping needs the gradient-norm scalar");
  return adam_launch(*p, (cudaStream_t)stream);
}
int dalle_b200_embed_fwd(const int64_t* ids, const float* weight, float* out, int batch, int seg_len, int n, int seg_off, int d, int vocab,
                         void* stream) {
  DB200_CHECK_ARG(ids && weight && out, "embed_fwd: null pointer");
  DB200_CHECK_ARG(batch >= 0 && seg_len >= 0 && n > 0 && seg_off >= 0 && seg_off + seg_len <= n && vocab > 0, "embed_fwd: bad geometry");
  DB200_CHECK_ARG(d > 0 && d % 4 == 0 && aligned16(weight) && aligned16(out), "embed_fwd: d must be a multiple of 4, pointers 16-byte aligned");
  return embed_launch(false, reinterpret_cast<const long long*>(ids), weight, out, batch, seg_len, n, seg_off, d, vocab, (cudaStream_t)stream);
}
int dalle_b200_embed_bwd(const int64_t* ids, const float* d_out, float* dweight, int batch, int seg_len, int n, int seg_off, int d, int vocab,
                         void* stream) {
  DB200_CHECK_ARG(ids && d_out && dweight, "embed_bwd: null pointer");
  DB200_CHECK_ARG(batch >= 0 && seg_len >= 0 && n > 0 && seg_off >= 0 && seg_off + seg_len <= n && vocab > 0, "embed_bwd: bad geometry");
  DB200_CHECK_ARG(d > 0 && d % 4 == 0 && aligned16(d_out) && aligned16(dweight), "embed_bwd: d must be a multiple of 4, pointers 16-byte aligned");
  return embed_launch(true, reinterpret_cast<const long long*>(ids), d_out, dweight, batch, seg_len, n, seg_off, d, vocab, (cudaStream_t)stream);
}
int dalle_b200_axpby(const float* a, const float* b, float alpha, float* y, int64_t count, void* stream) {
  DB200_CHECK_ARG(a && b && y && count >= 0, "axpby: bad args");
  DB200_CHECK_ARG(aligned16(a) && aligned16(b) && aligned16(y), "axpby: alignment");
  return axpby_launch(a, b, alpha, y, count, (cudaStream_t)stream);
}

}  // extern "C"
