// Weight-streaming GEMM for M <= 32 rows (KV-cache decoding: one token per sequence).  acc[M,N] = sum_k A[m,k] * W[n,k], bf16 operands,
// both K-major, fp32 accumulation.
//
// At M = 16 a Linear layer is a pass over its weight matrix: 2 bytes of W per 32 flops, so HBM decides (25 MB of bf16 weights per C2
// layer = ~4 us at 6.5 TB/s) -- provided ALL SMs pull.  The tcgen05 kernel is built for 128-row tiles: at M = 16 it launches
// N / 128 or N / 256 CTAs (8 for the output projection), each streaming its weight slab alone: 13 - 20 us per GEMM, 56 % of a
// decoding step (profiles/r02_decode_step_launches_flat.txt).  CUDA cores cannot do it either (16 FMA per weight element = 100 TFLOP/s
// at HBM speed), so the math runs on mma.sync.m16n8k16: the 16 rows of A are exactly one A fragment.
//
// CTA = 8 warps = 16 output columns (two n8 tiles; for GEGLU the value tile j..j+7 and its gate tile H+j..H+j+7); the K range is cut
// into 8 contiguous slices, one per warp, so a CTA streams 16 weight rows end to end and N/16 (64 - 512) CTAs cover the machine.
// Per 32-wide K block a lane loads ONE 16-byte piece of a weight row (row = lane/4, 8 consecutive k at (lane%4)*8) and the matching
// pieces of A rows lane/4 and lane/4+8: those 8 + 8 + 8 values are the B and A fragments of TWO k16 steps under a permutation of k
// inside the block (a dot product does not care in which order k is visited, as long as A and B agree), so every global access is
// a 16-byte load and a weight row is read in 64-byte runs.  A (at most 16 x K bf16) is re-read by every CTA from L2.
// The 8 partial 16x16 accumulators of a CTA are summed through shared memory in a fixed order (deterministic), then the epilogue runs
// one thread per output element.
#include "common.cuh"

namespace db200 {

constexpr int SM_WARPS = 8, SM_THREADS = SM_WARPS * 32, SM_KBLK = 32;

__device__ __forceinline__ void mma_bf16_16816(float* c, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

struct SmallMArgs {
  const __nv_bfloat16* A; const __nv_bfloat16* W; int M, N, K;
  int epilogue;
  const float* bias;
  // STORE
  void* C; long long ldc; int c_dtype;
  // RESID
  const float* resid; const float* scale; float sign; __nv_bfloat16* y_out; float* out;
  // GEGLU
  __nv_bfloat16* u_out; __nv_bfloat16* h_out; int hidden;
};

// SM_UNROLL K blocks (16-byte loads of 2 weight rows + 2 A rows each) are issued back to back; the launcher picks a divisor of the block count
template <int SM_UNROLL>
__global__ void __launch_bounds__(SM_THREADS) gemm_smallm_kernel(SmallMArgs P) {
  __shared__ float red[SM_WARPS][16][17];
  __shared__ float fin[16][17];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const bool geglu = P.epilogue == DB200_EPI_GEGLU;
  // columns of the two n8 tiles
  const int col0 = geglu ? blockIdx.x * 8 : blockIdx.x * 16;
  const int col1 = geglu ? P.hidden + blockIdx.x * 8 : blockIdx.x * 16 + 8;
  const int kslice = P.K / SM_WARPS;                       // multiple of SM_KBLK (launcher checks K % 256 == 0)
  const long long k0 = (long long)warp * kslice + t * 8;
  const uint4* w0 = reinterpret_cast<const uint4*>(P.W + (long long)(col0 + g) * P.K + k0);
  const uint4* w1 = reinterpret_cast<const uint4*>(P.W + (long long)(col1 + g) * P.K + k0);
  const bool lo_ok = g < P.M, hi_ok = g + 8 < P.M;
  const uint4* alo = reinterpret_cast<const uint4*>(P.A + (long long)(lo_ok ? g : 0) * P.K + k0);
  const uint4* ahi = reinterpret_cast<const uint4*>(P.A + (long long)(hi_ok ? g + 8 : 0) * P.K + k0);
  const uint4 zero4 = make_uint4(0u, 0u, 0u, 0u);
  float c0[4] = {0.f, 0.f, 0.f, 0.f}, c1[4] = {0.f, 0.f, 0.f, 0.f};
  const int nblk = kslice / SM_KBLK;                       // 16-byte pieces are SM_KBLK * 2 / 16 = 4 uint4 apart
  for (int b0 = 0; b0 < nblk; b0 += SM_UNROLL) {           // nblk % SM_UNROLL == 0
    uint4 bw0[SM_UNROLL], bw1[SM_UNROLL], al[SM_UNROLL], ah[SM_UNROLL];
#pragma unroll
    for (int u = 0; u < SM_UNROLL; ++u) {
      bw0[u] = __ldg(w0 + (b0 + u) * 4);
      bw1[u] = __ldg(w1 + (b0 + u) * 4);
      al[u] = __ldg(alo + (b0 + u) * 4);
      ah[u] = __ldg(ahi + (b0 + u) * 4);
    }
#pragma unroll
    for (int u = 0; u < SM_UNROLL; ++u) {
      const uint4 l = lo_ok ? al[u] : zero4, h = hi_ok ? ah[u] : zero4;
      // k16 step 0 = pieces .x (logical k 2t, 2t+1) and .y (logical k 2t+8, 2t+9); step 1 = .z and .w
      mma_bf16_16816(c0, l.x, h.x, l.y, h.y, bw0[u].x, bw0[u].y);
      mma_bf16_16816(c1, l.x, h.x, l.y, h.y, bw1[u].x, bw1[u].y);
      mma_bf16_16816(c0, l.z, h.z, l.w, h.w, bw0[u].z, bw0[u].w);
      mma_bf16_16816(c1, l.z, h.z, l.w, h.w, bw1[u].z, bw1[u].w);
    }
  }
  // accumulator fragment: c[0], c[1] = row g, columns 2t, 2t+1 ; c[2], c[3] = row g+8
  red[warp][g][2 * t] = c0[0]; red[warp][g][2 * t + 1] = c0[1];
  red[warp][g + 8][2 * t] = c0[2]; red[warp][g + 8][2 * t + 1] = c0[3];
  red[warp][g][8 + 2 * t] = c1[0]; red[warp][g][8 + 2 * t + 1] = c1[1];
  red[warp][g + 8][8 + 2 * t] = c1[2]; red[warp][g + 8][8 + 2 * t + 1] = c1[3];
  __syncthreads();
  const int m = tid >> 4, c = tid & 15;
  float acc = 0.f;
#pragma unroll
  for (int w = 0; w < SM_WARPS; ++w) acc += red[w][m][c];
  const int n = c < 8 ? col0 + c : col1 + (c - 8);
  if (P.bias) acc += __ldg(P.bias + n);
  if (geglu) {
    fin[m][c] = acc;
    __syncthreads();
    if (m < P.M) {
      if (P.u_out) P.u_out[(long long)m * P.N + n] = __float2bfloat16_rn(acc);
      if (c < 8) P.h_out[(long long)m * P.hidden + n] = __float2bfloat16_rn(fin[m][c] * gelu_erf(fin[m][c + 8]));
    }
    return;
  }
  if (m >= P.M) return;
  if (P.epilogue == DB200_EPI_STORE) {
    const long long o = (long long)m * P.ldc + n;
    if (P.c_dtype == DB200_F32) reinterpret_cast<float*>(P.C)[o] = acc;
    else reinterpret_cast<__nv_bfloat16*>(P.C)[o] = __float2bfloat16_rn(acc);
  } else {                                                 // RESID
    const long long o = (long long)m * P.N + n;
    if (P.y_out) P.y_out[o] = __float2bfloat16_rn(acc);
    const float r = P.resid ? P.resid[o] : 0.f;
    const float s = P.scale ? __ldg(P.scale + n) : 1.f;
    P.out[o] = r + P.sign * s * acc;
  }
}

// 17 <= M <= 32 rows (classifier-free guidance decodes the conditional and the unconditional stream as ONE batch of 2b rows): the same
// CTA layout and weight stream with a second A fragment (rows 16-31).  Every loaded B fragment feeds two mma.sync, so a CTA reads
// exactly the weight bytes of the 16-row kernel.  A separate kernel rather than a fragment-count template parameter of the one
// above, so that the M <= 16 kernel (unguided decoding) compiles to the same code as before.
template <int SM_UNROLL>
__global__ void __launch_bounds__(SM_THREADS) gemm_smallm32_kernel(SmallMArgs P) {
  __shared__ float red[SM_WARPS][32][17];
  __shared__ float fin[32][17];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const bool geglu = P.epilogue == DB200_EPI_GEGLU;
  const int col0 = geglu ? blockIdx.x * 8 : blockIdx.x * 16;
  const int col1 = geglu ? P.hidden + blockIdx.x * 8 : blockIdx.x * 16 + 8;
  const int kslice = P.K / SM_WARPS;
  const long long k0 = (long long)warp * kslice + t * 8;
  const uint4* w0 = reinterpret_cast<const uint4*>(P.W + (long long)(col0 + g) * P.K + k0);
  const uint4* w1 = reinterpret_cast<const uint4*>(P.W + (long long)(col1 + g) * P.K + k0);
  // A rows g, g+8 (fragment 0) and g+16, g+24 (fragment 1); rows 0..15 always exist (M > 16)
  const bool ok2 = g + 16 < P.M, ok3 = g + 24 < P.M;
  const uint4* a0 = reinterpret_cast<const uint4*>(P.A + (long long)g * P.K + k0);
  const uint4* a1 = reinterpret_cast<const uint4*>(P.A + (long long)(g + 8) * P.K + k0);
  const uint4* a2 = reinterpret_cast<const uint4*>(P.A + (long long)(ok2 ? g + 16 : 0) * P.K + k0);
  const uint4* a3 = reinterpret_cast<const uint4*>(P.A + (long long)(ok3 ? g + 24 : 0) * P.K + k0);
  const uint4 zero4 = make_uint4(0u, 0u, 0u, 0u);
  float c00[4] = {0.f, 0.f, 0.f, 0.f}, c10[4] = {0.f, 0.f, 0.f, 0.f};      // c<n tile><fragment>
  float c01[4] = {0.f, 0.f, 0.f, 0.f}, c11[4] = {0.f, 0.f, 0.f, 0.f};
  const int nblk = kslice / SM_KBLK;
  for (int b0 = 0; b0 < nblk; b0 += SM_UNROLL) {
    uint4 bw0[SM_UNROLL], bw1[SM_UNROLL], r0[SM_UNROLL], r1[SM_UNROLL], r2[SM_UNROLL], r3[SM_UNROLL];
#pragma unroll
    for (int u = 0; u < SM_UNROLL; ++u) {
      bw0[u] = __ldg(w0 + (b0 + u) * 4);
      bw1[u] = __ldg(w1 + (b0 + u) * 4);
      r0[u] = __ldg(a0 + (b0 + u) * 4);
      r1[u] = __ldg(a1 + (b0 + u) * 4);
      r2[u] = __ldg(a2 + (b0 + u) * 4);
      r3[u] = __ldg(a3 + (b0 + u) * 4);
    }
#pragma unroll
    for (int u = 0; u < SM_UNROLL; ++u) {
      const uint4 l0 = r0[u], h0 = r1[u], l1 = ok2 ? r2[u] : zero4, h1 = ok3 ? r3[u] : zero4;
      mma_bf16_16816(c00, l0.x, h0.x, l0.y, h0.y, bw0[u].x, bw0[u].y);
      mma_bf16_16816(c10, l0.x, h0.x, l0.y, h0.y, bw1[u].x, bw1[u].y);
      mma_bf16_16816(c01, l1.x, h1.x, l1.y, h1.y, bw0[u].x, bw0[u].y);
      mma_bf16_16816(c11, l1.x, h1.x, l1.y, h1.y, bw1[u].x, bw1[u].y);
      mma_bf16_16816(c00, l0.z, h0.z, l0.w, h0.w, bw0[u].z, bw0[u].w);
      mma_bf16_16816(c10, l0.z, h0.z, l0.w, h0.w, bw1[u].z, bw1[u].w);
      mma_bf16_16816(c01, l1.z, h1.z, l1.w, h1.w, bw0[u].z, bw0[u].w);
      mma_bf16_16816(c11, l1.z, h1.z, l1.w, h1.w, bw1[u].z, bw1[u].w);
    }
  }
  red[warp][g][2 * t] = c00[0]; red[warp][g][2 * t + 1] = c00[1];
  red[warp][g + 8][2 * t] = c00[2]; red[warp][g + 8][2 * t + 1] = c00[3];
  red[warp][g][8 + 2 * t] = c10[0]; red[warp][g][8 + 2 * t + 1] = c10[1];
  red[warp][g + 8][8 + 2 * t] = c10[2]; red[warp][g + 8][8 + 2 * t + 1] = c10[3];
  red[warp][g + 16][2 * t] = c01[0]; red[warp][g + 16][2 * t + 1] = c01[1];
  red[warp][g + 24][2 * t] = c01[2]; red[warp][g + 24][2 * t + 1] = c01[3];
  red[warp][g + 16][8 + 2 * t] = c11[0]; red[warp][g + 16][8 + 2 * t + 1] = c11[1];
  red[warp][g + 24][8 + 2 * t] = c11[2]; red[warp][g + 24][8 + 2 * t + 1] = c11[3];
  __syncthreads();
  // thread -> column c of rows m and m + 16 (the same fixed-order reduction as the 16-row kernel)
  const int m = tid >> 4, c = tid & 15;
  float acc_lo = 0.f, acc_hi = 0.f;
#pragma unroll
  for (int w = 0; w < SM_WARPS; ++w) { acc_lo += red[w][m][c]; acc_hi += red[w][m + 16][c]; }
  const int n = c < 8 ? col0 + c : col1 + (c - 8);
  if (P.bias) { const float bv = __ldg(P.bias + n); acc_lo += bv; acc_hi += bv; }
  if (geglu) {
    fin[m][c] = acc_lo;
    fin[m + 16][c] = acc_hi;
    __syncthreads();
    if (P.u_out) P.u_out[(long long)m * P.N + n] = __float2bfloat16_rn(acc_lo);
    if (c < 8) P.h_out[(long long)m * P.hidden + n] = __float2bfloat16_rn(fin[m][c] * gelu_erf(fin[m][c + 8]));
    if (m + 16 < P.M) {
      if (P.u_out) P.u_out[(long long)(m + 16) * P.N + n] = __float2bfloat16_rn(acc_hi);
      if (c < 8) P.h_out[(long long)(m + 16) * P.hidden + n] = __float2bfloat16_rn(fin[m + 16][c] * gelu_erf(fin[m + 16][c + 8]));
    }
    return;
  }
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    const int mm = m + 16 * half;
    const float acc = half ? acc_hi : acc_lo;
    if (mm >= P.M) break;
    if (P.epilogue == DB200_EPI_STORE) {
      const long long o = (long long)mm * P.ldc + n;
      if (P.c_dtype == DB200_F32) reinterpret_cast<float*>(P.C)[o] = acc;
      else reinterpret_cast<__nv_bfloat16*>(P.C)[o] = __float2bfloat16_rn(acc);
    } else {                                               // RESID
      const long long o = (long long)mm * P.N + n;
      if (P.y_out) P.y_out[o] = __float2bfloat16_rn(acc);
      const float r = P.resid ? P.resid[o] : 0.f;
      const float s = P.scale ? __ldg(P.scale + n) : 1.f;
      P.out[o] = r + P.sign * s * acc;
    }
  }
}

bool gemm_smallm_supported(const db200_gemm_params& p, const char** why) {
  const char* w = nullptr;
  if (p.dtype != DB200_BF16) w = "bf16 operands only";
  else if (p.M < 1 || p.M > 32) w = "1 <= M <= 32";
  else if (p.a_mn_major || p.b_mn_major) w = "both operands must be K-major";
  else if (p.K % (SM_WARPS * SM_KBLK) != 0) w = "K must be a multiple of 256";
  else if (p.lda != p.K || p.ldb != p.K) w = "operands must be dense (lda = ldb = K)";
  else if ((reinterpret_cast<uintptr_t>(p.A) | reinterpret_cast<uintptr_t>(p.B)) & 15) w = "operands must be 16-byte aligned";
  else if (p.epilogue == DB200_EPI_STORE) {
    if (p.N % 16) w = "N must be a multiple of 16";
    else if (p.split_k_ok || p.C_multicast) w = "no split-K / multicast accumulation";
  } else if (p.epilogue == DB200_EPI_RESID) {
    if (p.N % 16) w = "N must be a multiple of 16";
  } else if (p.epilogue == DB200_EPI_GEGLU) {
    if (p.hidden % 8) w = "hidden must be a multiple of 8";
  } else w = "epilogue not implemented for the small-M kernel (STORE, RESID, GEGLU are)";
  if (why) *why = w ? w : "";
  return w == nullptr;
}

int gemm_smallm_launch(const db200_gemm_params& p, cudaStream_t st) {
  SmallMArgs a;
  a.A = reinterpret_cast<const __nv_bfloat16*>(p.A); a.W = reinterpret_cast<const __nv_bfloat16*>(p.B);
  a.M = p.M; a.N = p.N; a.K = p.K; a.epilogue = p.epilogue; a.bias = p.bias;
  a.C = p.C; a.ldc = p.ldc; a.c_dtype = p.c_dtype;
  a.resid = p.resid; a.scale = p.scale; a.sign = p.sign; a.y_out = reinterpret_cast<__nv_bfloat16*>(p.y_out); a.out = p.out;
  a.u_out = reinterpret_cast<__nv_bfloat16*>(p.u_out); a.h_out = reinterpret_cast<__nv_bfloat16*>(p.h_out); a.hidden = p.hidden;
  const int grid = p.epilogue == DB200_EPI_GEGLU ? p.hidden / 8 : p.N / 16;
  const int nblk = p.K / (SM_WARPS * SM_KBLK);
  if (p.M > 16) {
    if (nblk % 4 == 0) gemm_smallm32_kernel<4><<<grid, SM_THREADS, 0, st>>>(a);
    else if (nblk % 2 == 0) gemm_smallm32_kernel<2><<<grid, SM_THREADS, 0, st>>>(a);
    else gemm_smallm32_kernel<1><<<grid, SM_THREADS, 0, st>>>(a);
    DB200_LAUNCH_OK("gemm_smallm32_kernel");
    return DB200_OK;
  }
  if (nblk % 4 == 0) gemm_smallm_kernel<4><<<grid, SM_THREADS, 0, st>>>(a);
  else if (nblk % 2 == 0) gemm_smallm_kernel<2><<<grid, SM_THREADS, 0, st>>>(a);
  else gemm_smallm_kernel<1><<<grid, SM_THREADS, 0, st>>>(a);
  DB200_LAUNCH_OK("gemm_smallm_kernel");
  return DB200_OK;
}

}  // namespace db200
