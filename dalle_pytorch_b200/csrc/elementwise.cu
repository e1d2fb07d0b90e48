// HBM-bound glue kernels of the DALL-E block: LayerNorm + token-shift (forward and backward), LayerScale /
// residual backward, column sums, casts.  Each is one pass over its tensor with 16-byte accesses.
#include <cmath>

#include "common.cuh"
#include "epilogue.cuh"
#include "tc_common.cuh"

namespace db200 {

namespace {

constexpr int LN_THREADS = 128;

__device__ __forceinline__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();                         // protect `red` against the previous use
  if (l == 0) red[w] = v;
  __syncthreads();
  float t = 0.f;
  const int nw = blockDim.x >> 5;
  for (int i = 0; i < nw; ++i) t += red[i];
  return t;
}

// Where does channel c of the (LayerNorm-ed) token at position p end up after PreShiftToken?
// transformer.py:165-186: text tokens shift their first half to p+1; image token (r,c) sends its first
// quarter to the token below (r+1,c) and its second quarter to the right neighbour (r,c+1); -1 = dropped.
__device__ __forceinline__ int shift_dest(int p, int c, int n, int d, int text_len, int fmap, int do_shift) {
  if (!do_shift || c >= (d >> 1)) return p;
  if (p < text_len) return (p + 1 < text_len) ? p + 1 : -1;
  const int q = p - text_len;
  const int r = q / fmap, cc = q - r * fmap;
  if (c < (d >> 2)) return (r + 1 < fmap && p + fmap < n) ? p + fmap : -1;
  return (cc + 1 < fmap && p + 1 < n) ? p + 1 : -1;
}

// Same mapping resolved ONCE per token row (one integer division), then applied per channel range with compares only: the
// streaming kernels below are issue-bound, not HBM-bound, if the division is repeated for every 4-channel chunk (ncu, r01).
struct ShiftRow {
  int dest_q1, dest_q2;     // where channels [0,d/4) / [d/4,d/2) of this row go (-1 = dropped); channels >= d/2 stay
  bool zero_q1, zero_q2;    // does this row receive nothing in those ranges (so zeros must be written)
  int self;
};
__device__ __forceinline__ ShiftRow make_shift_row(int p, int n, int text_len, int fmap, int do_shift) {
  ShiftRow s;
  s.self = p;
  if (!do_shift) { s.dest_q1 = s.dest_q2 = p; s.zero_q1 = s.zero_q2 = false; return s; }
  if (p < text_len) {
    s.dest_q1 = s.dest_q2 = (p + 1 < text_len) ? p + 1 : -1;
    s.zero_q1 = s.zero_q2 = (p == 0);
  } else {
    const int q = p - text_len;
    const int r = q / fmap, cc = q - r * fmap;
    s.dest_q1 = (r + 1 < fmap && p + fmap < n) ? p + fmap : -1;
    s.dest_q2 = (cc + 1 < fmap && p + 1 < n) ? p + 1 : -1;
    s.zero_q1 = (r == 0);
    s.zero_q2 = (cc == 0);
  }
  return s;
}
__device__ __forceinline__ int shift_row_dest(const ShiftRow& s, int c, int d) { return c >= (d >> 1) ? s.self : (c < (d >> 2) ? s.dest_q1 : s.dest_q2); }

template <typename TO>
__global__ void __launch_bounds__(LN_THREADS) ln_shift_fwd_kernel(db200_ln_shift_fwd_params P) {
  extern __shared__ float row[];
  __shared__ float red[LN_THREADS / 32];
  const int r = blockIdx.x;
  const int n = P.n, d = P.d;
  const int b = r / n, p = r - b * n;
  const float* xr = P.x + (long long)r * d;
  float s = 0.f;
  for (int c = threadIdx.x * 4; c < d; c += LN_THREADS * 4) {
    const float4 v = *reinterpret_cast<const float4*>(xr + c);
    *reinterpret_cast<float4*>(row + c) = v;
    s += (v.x + v.y) + (v.z + v.w);
  }
  float mean = 0.f, rstd = 1.f;
  if (P.do_ln) {
    mean = block_sum(s, red) / d;
    float q = 0.f;
    for (int c = threadIdx.x * 4; c < d; c += LN_THREADS * 4) {
      const float4 v = *reinterpret_cast<const float4*>(row + c);
      const float a0 = v.x - mean, a1 = v.y - mean, a2 = v.z - mean, a3 = v.w - mean;
      q += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
    }
    const float var = block_sum(q, red) / d;
    rstd = 1.0f / sqrtf(var + P.eps);
    if (threadIdx.x == 0) { P.mean[r] = mean; P.rstd[r] = rstd; }
  }
  TO* out = reinterpret_cast<TO*>(P.out);
  const long long brow = (long long)b * n;
  for (int c = threadIdx.x * 4; c < d; c += LN_THREADS * 4) {
    float4 v = *reinterpret_cast<const float4*>(row + c);
    if (P.do_ln) {
      const float4 g = *reinterpret_cast<const float4*>(P.gamma + c);
      const float4 be = *reinterpret_cast<const float4*>(P.beta + c);
      v.x = (v.x - mean) * rstd * g.x + be.x;
      v.y = (v.y - mean) * rstd * g.y + be.y;
      v.z = (v.z - mean) * rstd * g.z + be.z;
      v.w = (v.w - mean) * rstd * g.w + be.w;
    }
    const int dest = shift_dest(p, c, n, d, P.text_len, P.fmap, P.do_shift);
    if (dest >= 0) {
      TO* o = out + (brow + dest) * d + c;
      store2<TO>(o, v.x, v.y);
      store2<TO>(o + 2, v.z, v.w);
    }
    if (P.do_shift && c < (d >> 1)) {
      // positions that receive nothing get zeros (F.pad in transformer.py:172,178-179)
      bool zero;
      if (p < P.text_len) zero = (p == 0);
      else {
        const int q = p - P.text_len;
        const int rr = q / P.fmap, cc = q - rr * P.fmap;
        zero = (c < (d >> 2)) ? (rr == 0) : (cc == 0);
      }
      if (zero) {
        TO* o = out + (brow + p) * d + c;
        store2<TO>(o, 0.f, 0.f);
        store2<TO>(o + 2, 0.f, 0.f);
      }
    }
  }
}

template <typename TI>
__global__ void __launch_bounds__(LN_THREADS) ln_shift_bwd_kernel(db200_ln_shift_bwd_params P) {
  extern __shared__ float sm[];
  __shared__ float red[LN_THREADS / 32];
  const int n = P.n, d = P.d;
  float* dy = sm;             // [d] gradient w.r.t. the LN output of this row (after un-shifting)
  float* xh = sm + d;         // [d] x_hat
  float* accg = sm + 2 * d;   // [d] dgamma partial
  float* accb = sm + 3 * d;   // [d] dbeta partial
  for (int c = threadIdx.x; c < d; c += LN_THREADS) { accg[c] = 0.f; accb[c] = 0.f; }
  __syncthreads();            // the accumulation below uses a different thread <-> channel mapping (compute-sanitizer racecheck, r02)
  const TI* dA = reinterpret_cast<const TI*>(P.d_out);
  const int rows = P.batch * n;
  for (int r = blockIdx.x; r < rows; r += gridDim.x) {
    const int b = r / n, p = r - b * n;
    const long long brow = (long long)b * n;
    const float* xr = P.x + (long long)r * d;
    float mean = 0.f, rstd = 1.f;
    if (P.do_ln) { mean = P.mean[r]; rstd = P.rstd[r]; }
    float s1 = 0.f, s2 = 0.f;
    for (int c = threadIdx.x * 4; c < d; c += LN_THREADS * 4) {
      const int src = shift_dest(p, c, n, d, P.text_len, P.fmap, P.do_shift);
      float g0 = 0.f, g1 = 0.f, g2 = 0.f, g3 = 0.f;
      if (src >= 0) {
        const TI* gp = dA + (brow + src) * d + c;
        const float2 a = load2<TI>(gp), bb = load2<TI>(gp + 2);
        g0 = a.x; g1 = a.y; g2 = bb.x; g3 = bb.y;
      }
      if (P.do_ln) {
        const float4 xv = *reinterpret_cast<const float4*>(xr + c);
        const float4 ga = *reinterpret_cast<const float4*>(P.gamma + c);
        const float h0 = (xv.x - mean) * rstd, h1 = (xv.y - mean) * rstd, h2 = (xv.z - mean) * rstd, h3 = (xv.w - mean) * rstd;
        accg[c] += g0 * h0; accg[c + 1] += g1 * h1; accg[c + 2] += g2 * h2; accg[c + 3] += g3 * h3;
        accb[c] += g0; accb[c + 1] += g1; accb[c + 2] += g2; accb[c + 3] += g3;
        g0 *= ga.x; g1 *= ga.y; g2 *= ga.z; g3 *= ga.w;
        s1 += (g0 + g1) + (g2 + g3);
        s2 += (g0 * h0 + g1 * h1) + (g2 * h2 + g3 * h3);
        *reinterpret_cast<float4*>(xh + c) = make_float4(h0, h1, h2, h3);
      }
      *reinterpret_cast<float4*>(dy + c) = make_float4(g0, g1, g2, g3);
    }
    float m1 = 0.f, m2 = 0.f;
    if (P.do_ln) {
      m1 = block_sum(s1, red) / d;
      m2 = block_sum(s2, red) / d;
    }
    float* dxr = P.dx + (long long)r * d;
    const float* dr = P.dres ? P.dres + (long long)r * d : nullptr;
    for (int c = threadIdx.x * 4; c < d; c += LN_THREADS * 4) {
      float4 g = *reinterpret_cast<const float4*>(dy + c);
      if (P.do_ln) {
        const float4 h = *reinterpret_cast<const float4*>(xh + c);
        g.x = rstd * (g.x - m1 - h.x * m2);
        g.y = rstd * (g.y - m1 - h.y * m2);
        g.z = rstd * (g.z - m1 - h.z * m2);
        g.w = rstd * (g.w - m1 - h.w * m2);
      }
      if (dr) {
        const float4 e = *reinterpret_cast<const float4*>(dr + c);
        g.x += e.x; g.y += e.y; g.z += e.z; g.w += e.w;
      }
      *reinterpret_cast<float4*>(dxr + c) = g;
    }
    // each thread only ever touches its own channels of dy/xh/accg/accb -> no barrier needed between rows
  }
  if (P.do_ln && P.dgamma) {
    // same thread<->channel ownership as above
    for (int c = threadIdx.x * 4; c < d; c += LN_THREADS * 4) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        atomicAdd(P.dgamma + c + j, accg[c + j]);
        atomicAdd(P.dbeta + c + j, accb[c + j]);
      }
    }
  }
}


// =====================================================================================================================
// Warp-per-row variants for d = 128 * NCH (every benchmark configuration): the whole row lives in registers (4*NCH floats per
// lane), all reductions are warp shuffles (no block barriers), every global access is a contiguous 256-512 B segment per
// warp instruction.  These are the kernels that run in C2..C5; the CTA-per-row kernels above cover arbitrary d.
// =====================================================================================================================
constexpr int WR_WARPS = 8;

template <typename TO, int NCH>
__global__ void __launch_bounds__(WR_WARPS * 32) ln_shift_fwd_warp_kernel(db200_ln_shift_fwd_params P) {
  pdl_launch();
  pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rows = P.batch * P.n;
  const int r = blockIdx.x * WR_WARPS + warp;
  if (r >= rows) return;
  const int n = P.n, d = P.d;
  const int b = r / n, p = r - b * n;
  const float* xr = P.x + (long long)r * d;
  float4 v[NCH];
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < NCH; ++k) {
    v[k] = *reinterpret_cast<const float4*>(xr + k * 128 + lane * 4);
    s += (v[k].x + v[k].y) + (v[k].z + v[k].w);
  }
  float mean = 0.f, rstd = 1.f;
  if (P.do_ln) {
    mean = warp_sum(s) / d;
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      const float a0 = v[k].x - mean, a1 = v[k].y - mean, a2 = v[k].z - mean, a3 = v[k].w - mean;
      q += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
    }
    rstd = 1.0f / sqrtf(warp_sum(q) / d + P.eps);
    if (lane == 0) { P.mean[r] = mean; P.rstd[r] = rstd; }
  }
  TO* out = reinterpret_cast<TO*>(P.out);
  const long long brow = (long long)b * n;
  const ShiftRow sr = make_shift_row(p, n, P.text_len, P.fmap, P.do_shift);
#pragma unroll
  for (int k = 0; k < NCH; ++k) {
    const int c = k * 128 + lane * 4;
    float4 y = v[k];
    if (P.do_ln) {
      const float4 g = __ldg(reinterpret_cast<const float4*>(P.gamma + c));
      const float4 be = __ldg(reinterpret_cast<const float4*>(P.beta + c));
      y.x = (y.x - mean) * rstd * g.x + be.x;
      y.y = (y.y - mean) * rstd * g.y + be.y;
      y.z = (y.z - mean) * rstd * g.z + be.z;
      y.w = (y.w - mean) * rstd * g.w + be.w;
    }
    const int dest = shift_row_dest(sr, c, d);
    if (dest >= 0) {
      TO* o = out + (brow + dest) * d + c;
      store2<TO>(o, y.x, y.y);
      store2<TO>(o + 2, y.z, y.w);
    }
    if (c < (d >> 1) && ((c < (d >> 2)) ? sr.zero_q1 : sr.zero_q2)) {
      TO* o = out + (brow + p) * d + c;
      store2<TO>(o, 0.f, 0.f);
      store2<TO>(o + 2, 0.f, 0.f);
    }
  }
}

// LayerNorm(+shift) backward is split in two streaming kernels so that neither needs many registers:
//   (1) dx   : warp per row, single pass, row gradient and x_hat in registers (no cross-row state)  -> high occupancy
//   (2) dgamma/dbeta : thread = 4 channels, block = 1024 channels x SLAB_ROWS rows, register partial sums, one atomic per
//       channel and block.  (2) re-reads dA and x (126 MB at C2, ~20 us) which is cheaper than carrying 2*d/32 accumulators
//       per lane through (1).
template <typename TI, int NCH>
__global__ void __launch_bounds__(WR_WARPS * 32, 3) ln_shift_bwd_dx_kernel(db200_ln_shift_bwd_params P) {
  // dgamma / dbeta partials of the whole (persistent) block live in shared memory; lanes add into bank-conflict-free slots
  // ([k][j][lane]) with RED.shared, and the block issues ONE global atomic per channel at the end.
  extern __shared__ float sm[];          // [2][d]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = P.n, d = P.d;
  const int rows = P.batch * n;
  const bool want_p = P.do_ln && P.dgamma != nullptr;
  if (want_p) {
    for (int c = threadIdx.x; c < 2 * d; c += blockDim.x) sm[c] = 0.f;
    __syncthreads();
  }
  const TI* __restrict__ dA = reinterpret_cast<const TI*>(P.d_out);
  for (int r = blockIdx.x * WR_WARPS + warp; r < rows; r += gridDim.x * WR_WARPS) {
    const int b = r / n, p = r - b * n;
    const long long brow = (long long)b * n;
    const float* __restrict__ xr = P.x + (long long)r * d;
    float mean = 0.f, rstd = 1.f;
    if (P.do_ln) { mean = P.mean[r]; rstd = P.rstd[r]; }
    float4 g[NCH], h[NCH];
    float s1 = 0.f, s2 = 0.f;
    const ShiftRow sr = make_shift_row(p, n, P.text_len, P.fmap, P.do_shift);
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      const int c = k * 128 + lane * 4;
      const int src = shift_row_dest(sr, c, d);
      g[k] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (src >= 0) {
        const TI* gp = dA + (brow + src) * d + c;
        const float2 a = load2<TI>(gp), bb = load2<TI>(gp + 2);
        g[k] = make_float4(a.x, a.y, bb.x, bb.y);
      }
      h[k] = P.do_ln ? *reinterpret_cast<const float4*>(xr + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if (P.do_ln) {
#pragma unroll
      for (int k = 0; k < NCH; ++k) {
        const int c = k * 128 + lane * 4;
        const float4 ga = __ldg(reinterpret_cast<const float4*>(P.gamma + c));
        h[k] = make_float4((h[k].x - mean) * rstd, (h[k].y - mean) * rstd, (h[k].z - mean) * rstd, (h[k].w - mean) * rstd);
        if (want_p) {
          float* sg = sm + (k * 4) * 32 + lane;
          float* sb = sm + d + (k * 4) * 32 + lane;
          atomicAdd(sg, g[k].x * h[k].x); atomicAdd(sg + 32, g[k].y * h[k].y); atomicAdd(sg + 64, g[k].z * h[k].z); atomicAdd(sg + 96, g[k].w * h[k].w);
          atomicAdd(sb, g[k].x); atomicAdd(sb + 32, g[k].y); atomicAdd(sb + 64, g[k].z); atomicAdd(sb + 96, g[k].w);
        }
        g[k].x *= ga.x; g[k].y *= ga.y; g[k].z *= ga.z; g[k].w *= ga.w;
        s1 += (g[k].x + g[k].y) + (g[k].z + g[k].w);
        s2 += (g[k].x * h[k].x + g[k].y * h[k].y) + (g[k].z * h[k].z + g[k].w * h[k].w);
      }
    }
    float m1 = 0.f, m2 = 0.f;
    if (P.do_ln) { m1 = warp_sum(s1) / d; m2 = warp_sum(s2) / d; }
    float* __restrict__ dxr = P.dx + (long long)r * d;
    const float* __restrict__ dr = P.dres ? P.dres + (long long)r * d : nullptr;
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      const int c = k * 128 + lane * 4;
      float4 o = g[k];
      if (P.do_ln) {
        o.x = rstd * (o.x - m1 - h[k].x * m2);
        o.y = rstd * (o.y - m1 - h[k].y * m2);
        o.z = rstd * (o.z - m1 - h[k].z * m2);
        o.w = rstd * (o.w - m1 - h[k].w * m2);
      }
      if (dr) {
        const float4 e = *reinterpret_cast<const float4*>(dr + c);
        o.x += e.x; o.y += e.y; o.z += e.z; o.w += e.w;
      }
      *reinterpret_cast<float4*>(dxr + c) = o;
    }
  }
  if (want_p) {
    __syncthreads();
    for (int i = threadIdx.x; i < d; i += blockDim.x) {
      // slot i = (k*4 + j)*32 + lane  <->  channel k*128 + lane*4 + j
      const int lane_i = i & 31, kj = i >> 5, k = kj >> 2, j = kj & 3;
      const int c = k * 128 + lane_i * 4 + j;
      atomicAdd(P.dgamma + c, sm[i]);
      atomicAdd(P.dbeta + c, sm[d + i]);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// LayerNorm(+shift) backward for d = 1024, bulk-copy staged.  The register-only kernel above tops out near 3 TB/s: a thread can
// hold ~160 bytes of loads in flight, so an SM never has much more than 100 KB outstanding, and HBM3e needs about twice that
// (its 64 shared-memory float atomics per row and lane also compile to ATOMS.CAST.SPIN compare-and-swap loops).
// Here one producer warp streams batches of R token rows (dA row assembled from up to three source rows of the token shift,
// x row, residual-gradient row) into a STAGES-deep shared-memory ring with cp.async.bulk + mbarrier transaction counts, so
// ~160 KB per SM are always in flight; eight consumer warps (warp w = channels [128w, 128w+128)) read their slice with
// conflict-free 8/16-byte LDS, keep dgamma / dbeta partials in registers for the whole kernel (a thread's channels never
// change) and exchange the two row statistics through 2*R*8 floats of shared memory and one named barrier per batch.
// ---------------------------------------------------------------------------------------------------------------------
using namespace tc;
constexpr int LT_R = 4;            // rows per stage
constexpr int LT_NW = 8;           // consumer warps per group (d = 1024)
constexpr int LT_GROUPS = 1;       // consumer groups taking alternate batches (2 measured no faster: the ring, not the consumers, paces the kernel)
constexpr int LT_THREADS = (LT_GROUPS * LT_NW + 1) * 32;
constexpr int LT_D = LT_NW * 128;
template <typename TI>
struct LnTmaSmem {
  static constexpr int G_ROW = LT_D * (int)sizeof(TI), X_ROW = LT_D * 4;
  static constexpr int Y_OFF = LT_R * (G_ROW + 2 * X_ROW);                  // upstream branch output rows (fused LayerScale adjoint)
  static constexpr int STAGE = LT_R * (2 * G_ROW + 2 * X_ROW);              // dA | x | dres | up_y
  static constexpr int STAGES = (sizeof(TI) == 2) ? 4 : 3;                  // 192 KB either way
  static constexpr int FLAG_OFF = STAGES * STAGE;                           // [STAGES][R][4] ints: q1 present, q2 present, row valid, pad
  static constexpr int PART_OFF = FLAG_OFF + STAGES * LT_R * 16;            // [GROUPS][2][2R][8] floats
  static constexpr int BAR_OFF = PART_OFF + LT_GROUPS * 2 * 2 * LT_R * LT_NW * 4;   // full[STAGES], empty[STAGES]
  static constexpr int TOTAL = BAR_OFF + 2 * STAGES * 8 + 16;
};

template <typename TI>
__global__ void __launch_bounds__(LT_THREADS, 1) ln_shift_bwd_tma_kernel(db200_ln_shift_bwd_params P) {
  pdl_launch();
  using L = LnTmaSmem<TI>;
  constexpr int R = LT_R, d = LT_D, STAGES = L::STAGES;
  extern __shared__ __align__(128) uint8_t smem[];
  int* flags = reinterpret_cast<int*>(smem + L::FLAG_OFF);
  const uint32_t full_bar = smem_u32(smem + L::BAR_OFF), empty_bar = full_bar + 8 * STAGES;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = P.n, rows = P.batch * n;
  const bool ln = P.do_ln != 0;
  const bool has_res = P.dres != nullptr;
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar + 8 * s, 1); mbar_init(empty_bar + 8 * s, LT_NW); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  pdl_wait();
  const int step = gridDim.x * R;

  if (warp == LT_GROUPS * LT_NW) {
    // ======================================= producer =======================================
    // One lane per (row, copy): lane = 6*i + j handles copy j of row i (j: 0 dA quarter 1, 1 dA quarter 2, 2 dA upper half,
    // 3 x, 4 dres, 5 upstream y).  A single issuing thread needs ~2-3 k cycles of dependent integer work per batch (divisions of the shift
    // geometry, 20 address computations) and was the bottleneck of the whole kernel; spread over 20 lanes it is ~10x shorter.
    // The transaction bytes are summed across the warp and posted by lane 0 (copies that complete before the expect_tx only
    // drive the tx-count negative for a moment; the phase cannot complete before lane 0's arrival).
    const TI* __restrict__ dA = reinterpret_cast<const TI*>(P.d_out);
    const int i = lane / 6, j = lane - i * 6;
    const bool active = lane < 6 * R;
    const bool has_up = P.up_dy != nullptr && P.up_y != nullptr;
    int s = 0; uint32_t ph = 0;
    for (int r0 = blockIdx.x * R; r0 < rows; r0 += step) {
      mbar_wait(empty_bar + 8 * s, ph ^ 1);
      uint8_t* st = smem + s * L::STAGE;
      const uint32_t fb = full_bar + 8 * s;
      uint32_t bytes = 0;
      const int r = r0 + i;
      if (active && r < rows) {
        const int b = r / n, p = r - b * n;
        const long long brow = (long long)b * n;
        const ShiftRow sr = make_shift_row(p, n, P.text_len, P.fmap, P.do_shift);
        const uint32_t gdst = smem_u32(st + i * L::G_ROW);
        if (j == 0) {
          int* fl = flags + (s * R + i) * 4;
          fl[0] = sr.dest_q1 >= 0; fl[1] = sr.dest_q2 >= 0; fl[2] = 1;
          if (sr.dest_q1 >= 0) { bytes = L::G_ROW / 4; bulk_load_1d(gdst, dA + (brow + sr.dest_q1) * d, bytes, fb); }
        } else if (j == 1) {
          if (sr.dest_q2 >= 0) { bytes = L::G_ROW / 4; bulk_load_1d(gdst + L::G_ROW / 4, dA + (brow + sr.dest_q2) * d + d / 4, bytes, fb); }
        } else if (j == 2) {
          bytes = L::G_ROW / 2; bulk_load_1d(gdst + L::G_ROW / 2, dA + (brow + p) * d + d / 2, bytes, fb);
        } else if (j == 3) {
          if (ln) { bytes = L::X_ROW; bulk_load_1d(smem_u32(st + R * L::G_ROW + i * L::X_ROW), P.x + (long long)r * d, bytes, fb); }
        } else if (j == 4) {
          if (has_res) { bytes = L::X_ROW; bulk_load_1d(smem_u32(st + R * (L::G_ROW + L::X_ROW) + i * L::X_ROW), P.dres + (long long)r * d, bytes, fb); }
        } else {
          if (has_up) { bytes = L::G_ROW; bulk_load_1d(smem_u32(st + L::Y_OFF + i * L::G_ROW), reinterpret_cast<const TI*>(P.up_y) + (long long)r * d, bytes, fb); }
        }
      } else if (active && j == 0) {
        flags[(s * R + i) * 4 + 2] = 0;                      // row past the end
      }
      const uint32_t total = __reduce_add_sync(0xffffffffu, bytes);
      __syncwarp();                                          // flag stores of all lanes are ordered before lane 0's (release) arrive
      if (lane == 0) mbar_expect_tx(fb, total);
      if (++s == STAGES) { s = 0; ph ^= 1; }
    }
    return;
  }

  // ======================================= consumers =======================================
  // Two groups of eight warps take alternate batches (the per-batch chain LDS -> shuffles -> barrier -> LDS -> STG is mostly
  // latency, so one group cannot drain the ring at HBM speed); each group has its own named barrier and statistics buffers.
  const int grp = warp / LT_NW, cw = warp - grp * LT_NW;
  float (*part)[2 * R][LT_NW] = reinterpret_cast<float (*)[2 * R][LT_NW]>(smem + L::PART_OFF) + grp * 2;
  const int c = cw * 128 + lane * 4;
  const bool want_p = ln && P.dgamma != nullptr;
  const float4 ga = ln ? __ldg(reinterpret_cast<const float4*>(P.gamma + c)) : make_float4(1.f, 1.f, 1.f, 1.f);
  float4 ag = make_float4(0.f, 0.f, 0.f, 0.f), ab = make_float4(0.f, 0.f, 0.f, 0.f);
  const int qsel = c >= (d >> 1) ? 2 : (c < (d >> 2) ? 0 : 1);      // flag index of this warp's channels (2 = always present)
  // fused upstream LayerScale adjoint (see db200_ln_shift_bwd_params::up_*)
  const bool up = P.up_dy != nullptr;
  const bool up_has_y = up && P.up_y != nullptr;
  float4 usc = make_float4(P.up_sign, P.up_sign, P.up_sign, P.up_sign);
  if (up && P.up_scale) { const float4 t = __ldg(reinterpret_cast<const float4*>(P.up_scale + c)); usc.x *= t.x; usc.y *= t.y; usc.z *= t.z; usc.w *= t.w; }
  float4 uds = make_float4(0.f, 0.f, 0.f, 0.f), udb = make_float4(0.f, 0.f, 0.f, 0.f);
  TI* __restrict__ up_dy = reinterpret_cast<TI*>(P.up_dy);
  int buf = 0;
  for (int k = grp; ; k += LT_GROUPS, buf ^= 1) {
    const int r0 = (blockIdx.x + k * (int)gridDim.x) * R;
    if (r0 >= rows) break;
    const int s = k % STAGES;
    const uint32_t ph = (k / STAGES) & 1;
    float mean[R], rstd[R];
#pragma unroll
    for (int i = 0; i < R; ++i) {            // tiny broadcast loads, issued before the wait
      const int r = r0 + i;
      mean[i] = 0.f; rstd[i] = 1.f;
      if (ln && r < rows) { mean[i] = __ldg(P.mean + r); rstd[i] = __ldg(P.rstd + r); }
    }
    mbar_wait(full_bar + 8 * s, ph);
    const uint8_t* st = smem + s * L::STAGE;
    const int* fl = flags + (s * R) * 4;
    float4 g[R], h[R], e[R];
#pragma unroll
    for (int i = 0; i < R; ++i) {
      g[i] = make_float4(0.f, 0.f, 0.f, 0.f); h[i] = g[i]; e[i] = g[i];
      const bool valid = fl[i * 4 + 2] != 0;
      const bool present = valid && (qsel == 2 || fl[i * 4 + qsel] != 0);
      if (present) {
        const TI* gp = reinterpret_cast<const TI*>(st + i * L::G_ROW) + c;
        const float2 a = load2<TI>(gp), bq = load2<TI>(gp + 2);
        g[i] = make_float4(a.x, a.y, bq.x, bq.y);
      }
      if (valid && ln) h[i] = *reinterpret_cast<const float4*>(st + R * L::G_ROW + i * L::X_ROW + c * 4);
      if (valid && has_res) e[i] = *reinterpret_cast<const float4*>(st + R * (L::G_ROW + L::X_ROW) + i * L::X_ROW + c * 4);
    }
    float4 uy[R];
#pragma unroll
    for (int i = 0; i < R; ++i) {
      uy[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (up_has_y && fl[i * 4 + 2] != 0) {
        const TI* yp = reinterpret_cast<const TI*>(st + L::Y_OFF + i * L::G_ROW) + c;
        const float2 a = load2<TI>(yp), bq = load2<TI>(yp + 2);
        uy[i] = make_float4(a.x, a.y, bq.x, bq.y);
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(empty_bar + 8 * s);       // stage consumed into registers
    if (ln) {
      float s1[R], s2[R];
#pragma unroll
      for (int i = 0; i < R; ++i) {
        h[i] = make_float4((h[i].x - mean[i]) * rstd[i], (h[i].y - mean[i]) * rstd[i], (h[i].z - mean[i]) * rstd[i], (h[i].w - mean[i]) * rstd[i]);
        if (want_p) {
          ag.x += g[i].x * h[i].x; ag.y += g[i].y * h[i].y; ag.z += g[i].z * h[i].z; ag.w += g[i].w * h[i].w;
          ab.x += g[i].x; ab.y += g[i].y; ab.z += g[i].z; ab.w += g[i].w;
        }
        g[i].x *= ga.x; g[i].y *= ga.y; g[i].z *= ga.z; g[i].w *= ga.w;
        s1[i] = (g[i].x + g[i].y) + (g[i].z + g[i].w);
        s2[i] = (g[i].x * h[i].x + g[i].y * h[i].y) + (g[i].z * h[i].z + g[i].w * h[i].w);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int i = 0; i < R; ++i) {
          s1[i] += __shfl_xor_sync(0xffffffffu, s1[i], o);
          s2[i] += __shfl_xor_sync(0xffffffffu, s2[i], o);
        }
      }
      if (lane == 0) {
#pragma unroll
        for (int i = 0; i < R; ++i) { part[buf][i][cw] = s1[i]; part[buf][R + i][cw] = s2[i]; }
      }
      asm volatile("bar.sync %0, %1;" ::"r"(1 + grp), "r"(LT_NW * 32) : "memory");
#pragma unroll
      for (int i = 0; i < R; ++i) {
        const float4 a0 = *reinterpret_cast<const float4*>(&part[buf][i][0]), a1 = *reinterpret_cast<const float4*>(&part[buf][i][4]);
        const float4 b0 = *reinterpret_cast<const float4*>(&part[buf][R + i][0]), b1 = *reinterpret_cast<const float4*>(&part[buf][R + i][4]);
        const float m1 = (((a0.x + a0.y) + (a0.z + a0.w)) + ((a1.x + a1.y) + (a1.z + a1.w))) * (1.0f / d);
        const float m2 = (((b0.x + b0.y) + (b0.z + b0.w)) + ((b1.x + b1.y) + (b1.z + b1.w))) * (1.0f / d);
        g[i].x = rstd[i] * (g[i].x - m1 - h[i].x * m2);
        g[i].y = rstd[i] * (g[i].y - m1 - h[i].y * m2);
        g[i].z = rstd[i] * (g[i].z - m1 - h[i].z * m2);
        g[i].w = rstd[i] * (g[i].w - m1 - h[i].w * m2);
      }
    }
#pragma unroll
    for (int i = 0; i < R; ++i) {
      const int r = r0 + i;
      if (r < rows) {
        const float4 o = make_float4(g[i].x + e[i].x, g[i].y + e[i].y, g[i].z + e[i].z, g[i].w + e[i].w);
        *reinterpret_cast<float4*>(P.dx + (long long)r * d + c) = o;
        if (up) {
          const float4 dy = make_float4(usc.x * o.x, usc.y * o.y, usc.z * o.z, usc.w * o.w);
          TI* dst = up_dy + (long long)r * d + c;
          store2<TI>(dst, dy.x, dy.y);
          store2<TI>(dst + 2, dy.z, dy.w);
          udb.x += dy.x; udb.y += dy.y; udb.z += dy.z; udb.w += dy.w;
          uds.x += P.up_sign * o.x * uy[i].x; uds.y += P.up_sign * o.y * uy[i].y;
          uds.z += P.up_sign * o.z * uy[i].z; uds.w += P.up_sign * o.w * uy[i].w;
        }
      }
    }
  }
  if (up && P.up_dbias) {
    atomicAdd(P.up_dbias + c, udb.x); atomicAdd(P.up_dbias + c + 1, udb.y); atomicAdd(P.up_dbias + c + 2, udb.z); atomicAdd(P.up_dbias + c + 3, udb.w);
  }
  if (up && P.up_dscale) {
    atomicAdd(P.up_dscale + c, uds.x); atomicAdd(P.up_dscale + c + 1, uds.y); atomicAdd(P.up_dscale + c + 2, uds.z); atomicAdd(P.up_dscale + c + 3, uds.w);
  }
  if (want_p) {
    atomicAdd(P.dgamma + c, ag.x); atomicAdd(P.dgamma + c + 1, ag.y); atomicAdd(P.dgamma + c + 2, ag.z); atomicAdd(P.dgamma + c + 3, ag.w);
    atomicAdd(P.dbeta + c, ab.x); atomicAdd(P.dbeta + c + 1, ab.y); atomicAdd(P.dbeta + c + 2, ab.z); atomicAdd(P.dbeta + c + 3, ab.w);
  }
}

constexpr int SLAB_ROWS = 32;
template <typename TI>
__global__ void __launch_bounds__(256) ln_shift_bwd_param_kernel(db200_ln_shift_bwd_params P) {
  const int c = (blockIdx.x * 256 + threadIdx.x) * 4;
  const int n = P.n, d = P.d;
  if (c >= d) return;
  const int rows = P.batch * n;
  const int r0 = blockIdx.y * SLAB_ROWS, r1 = min(rows, r0 + SLAB_ROWS);
  const TI* __restrict__ dA = reinterpret_cast<const TI*>(P.d_out);
  const float* __restrict__ x = P.x;
  float4 ag = make_float4(0.f, 0.f, 0.f, 0.f), ab = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int rb = r0; rb < r1; rb += 4) {
    float2 a[4], bb[4];
    float4 xv[4];
    float mean[4], rstd[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {          // all loads of four rows first
      const int r = rb + i;
      a[i] = make_float2(0.f, 0.f); bb[i] = make_float2(0.f, 0.f); xv[i] = make_float4(0.f, 0.f, 0.f, 0.f); mean[i] = 0.f; rstd[i] = 0.f;
      if (r < r1) {
        const int b = r / n, p = r - b * n;
        const int src = shift_row_dest(make_shift_row(p, n, P.text_len, P.fmap, P.do_shift), c, d);
        if (src >= 0) {
          const TI* gp = dA + ((long long)b * n + src) * d + c;
          a[i] = load2<TI>(gp); bb[i] = load2<TI>(gp + 2);
        }
        xv[i] = *reinterpret_cast<const float4*>(x + (long long)r * d + c);
        mean[i] = __ldg(P.mean + r); rstd[i] = __ldg(P.rstd + r);
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      ag.x += a[i].x * (xv[i].x - mean[i]) * rstd[i]; ag.y += a[i].y * (xv[i].y - mean[i]) * rstd[i];
      ag.z += bb[i].x * (xv[i].z - mean[i]) * rstd[i]; ag.w += bb[i].y * (xv[i].w - mean[i]) * rstd[i];
      ab.x += a[i].x; ab.y += a[i].y; ab.z += bb[i].x; ab.w += bb[i].y;
    }
  }
  atomicAdd(P.dgamma + c, ag.x); atomicAdd(P.dgamma + c + 1, ag.y); atomicAdd(P.dgamma + c + 2, ag.z); atomicAdd(P.dgamma + c + 3, ag.w);
  atomicAdd(P.dbeta + c, ab.x); atomicAdd(P.dbeta + c + 1, ab.y); atomicAdd(P.dbeta + c + 2, ab.z); atomicAdd(P.dbeta + c + 3, ab.w);
}

// scale_bwd, slab streaming: thread = 4 channels, block = 1024 channels x rows_per_block rows; LayerScale value and the partial
// sums live in 12 registers, so occupancy is high and four rows of loads are in flight per thread.
template <typename T>
__global__ void __launch_bounds__(256, 2) scale_bwd_slab_kernel(db200_scale_bwd_params P, int rows_per_block) {
  pdl_launch();
  pdl_wait();
  const int c = (blockIdx.x * 256 + threadIdx.x) * 4;
  const int d = P.d;
  if (c >= d) return;
  const int r0 = blockIdx.y * rows_per_block, r1 = min(P.rows, r0 + rows_per_block);
  float4 sc = make_float4(P.sign, P.sign, P.sign, P.sign);
  if (P.scale) { const float4 t = __ldg(reinterpret_cast<const float4*>(P.scale + c)); sc.x *= t.x; sc.y *= t.y; sc.z *= t.z; sc.w *= t.w; }
  const T* __restrict__ y = reinterpret_cast<const T*>(P.y);
  T* __restrict__ dy = reinterpret_cast<T*>(P.dy);
  const float* __restrict__ dout = P.d_out;
  const bool want_s = P.dscale != nullptr && y != nullptr;
  float4 as = make_float4(0.f, 0.f, 0.f, 0.f), ab = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int rb = r0; rb < r1; rb += 8) {
    float4 g[8];
    float2 y0[8], y1[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {          // all loads of eight rows first
      const long long off = (long long)(rb + i) * d + c;
      g[i] = make_float4(0.f, 0.f, 0.f, 0.f); y0[i] = make_float2(0.f, 0.f); y1[i] = make_float2(0.f, 0.f);
      if (rb + i < r1) {
        g[i] = *reinterpret_cast<const float4*>(dout + off);
        if (want_s) { y0[i] = load2<T>(y + off); y1[i] = load2<T>(y + off + 2); }
      }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (rb + i < r1) {
        const long long off = (long long)(rb + i) * d + c;
        const float o0 = sc.x * g[i].x, o1 = sc.y * g[i].y, o2 = sc.z * g[i].z, o3 = sc.w * g[i].w;
        store2<T>(dy + off, o0, o1);
        store2<T>(dy + off + 2, o2, o3);
        ab.x += o0; ab.y += o1; ab.z += o2; ab.w += o3;
        as.x += P.sign * g[i].x * y0[i].x; as.y += P.sign * g[i].y * y0[i].y; as.z += P.sign * g[i].z * y1[i].x; as.w += P.sign * g[i].w * y1[i].y;
      }
    }
  }
  if (P.dscale) { atomicAdd(P.dscale + c, as.x); atomicAdd(P.dscale + c + 1, as.y); atomicAdd(P.dscale + c + 2, as.z); atomicAdd(P.dscale + c + 3, as.w); }
  if (P.dbias) { atomicAdd(P.dbias + c, ab.x); atomicAdd(P.dbias + c + 1, ab.y); atomicAdd(P.dbias + c + 2, ab.z); atomicAdd(P.dbias + c + 3, ab.w); }
}

template <typename T>
__global__ void __launch_bounds__(256) scale_bwd_kernel(db200_scale_bwd_params P) {
  extern __shared__ float sm[];
  const int d = P.d;
  float* accs = sm;       // [d]
  float* accb = sm + d;   // [d]
  for (int c = threadIdx.x; c < 2 * d; c += blockDim.x) sm[c] = 0.f;
  // ownership: thread t owns channel pairs c = 2*t + k*2*blockDim
  const T* y = reinterpret_cast<const T*>(P.y);
  T* dy = reinterpret_cast<T*>(P.dy);
  for (int r = blockIdx.x; r < P.rows; r += gridDim.x) {
    const long long off = (long long)r * d;
    for (int c = threadIdx.x * 2; c < d; c += blockDim.x * 2) {
      const float2 g = *reinterpret_cast<const float2*>(P.d_out + off + c);
      float s0 = P.sign, s1 = P.sign;
      if (P.scale) { s0 *= P.scale[c]; s1 *= P.scale[c + 1]; }
      const float o0 = s0 * g.x, o1 = s1 * g.y;
      store2<T>(dy + off + c, o0, o1);
      // dbias accumulates exactly what the GEMMs will consume (the rounded value in bf16 mode is within tolerance;
      // keep the unrounded fp32 one for accuracy)
      accb[c] += o0; accb[c + 1] += o1;
      if (P.dscale && y) {
        const float2 yy = load2<T>(y + off + c);
        accs[c] += P.sign * g.x * yy.x; accs[c + 1] += P.sign * g.y * yy.y;
      }
    }
  }
  for (int c = threadIdx.x * 2; c < d; c += blockDim.x * 2) {
    if (P.dscale) { atomicAdd(P.dscale + c, accs[c]); atomicAdd(P.dscale + c + 1, accs[c + 1]); }
    if (P.dbias) { atomicAdd(P.dbias + c, accb[c]); atomicAdd(P.dbias + c + 1, accb[c + 1]); }
  }
}

// GEGLU adjoint as one streaming pass (transformer.py:106-109 autograd): du = [dh*gelu(g) | dh*a*gelu'(g)], plus the column
// sums of du (= gradient of net.0.bias) accumulated on the fly.  Thread = 8 hidden columns, block = 2048 columns x rows_per_block rows
// (host-chosen so that the grid is whole waves of resident CTAs, see balanced_rows_per_block).
template <typename T>
__global__ void __launch_bounds__(256, 4) geglu_bwd_kernel(const T* __restrict__ dh, const T* __restrict__ u, T* __restrict__ du,
                                                        float* __restrict__ dbias, int rows, int hidden, int rows_per_block) {
  pdl_launch();
  pdl_wait();
  const int j = (blockIdx.x * 256 + threadIdx.x) * 8;
  if (j >= hidden) return;
  const int r0 = blockIdx.y * rows_per_block, r1 = min(rows, r0 + rows_per_block);
  float sa[8], sg[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { sa[i] = 0.f; sg[i] = 0.f; }
#pragma unroll 4
  for (int r = r0; r < r1; ++r) {
    float d[8], a[8], g[8], da[8], dg[8];
    Vec8<T>::load(dh + (long long)r * hidden + j, d);
    Vec8<T>::load(u + (long long)r * 2 * hidden + j, a);
    Vec8<T>::load(u + (long long)r * 2 * hidden + hidden + j, g);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float f, df;
      gelu_pair<T>(g[i], f, df);
      da[i] = d[i] * f;
      dg[i] = d[i] * a[i] * df;
      sa[i] += da[i];
      sg[i] += dg[i];
    }
    Vec8<T>::store(du + (long long)r * 2 * hidden + j, da);
    Vec8<T>::store(du + (long long)r * 2 * hidden + hidden + j, dg);
  }
  if (dbias) {
#pragma unroll
    for (int i = 0; i < 8; ++i) { atomicAdd(dbias + j + i, sa[i]); atomicAdd(dbias + hidden + j + i, sg[i]); }
  }
}

// ---- logits head: cross-entropy over rows of [rows, vocab] logits (dalle_pytorch.py:667-670) -----------------------------
// One 256-thread block per row, single pass with per-thread online (max, sum) pairs merged by shuffles: the logits are read
// once.  loss_acc += coef * (lse - logit[label]);  row_lse is kept for the backward pass.
__device__ __forceinline__ void ms_merge(float& m, float& s, float m2, float s2) {
  const float mn = fmaxf(m, m2);
  s = s * __expf(m - mn) + s2 * __expf(m2 - mn);
  m = mn;
}
template <typename T>
__global__ void __launch_bounds__(256) ce_fwd_kernel(const T* __restrict__ logits, const long long* __restrict__ labels, int vocab,
                                                     float coef, float* __restrict__ row_lse, float* __restrict__ loss_acc) {
  __shared__ float sm_m[8], sm_s[8];
  const int r = blockIdx.x;
  const T* row = logits + (long long)r * vocab;
  float m = -1.0e30f, s = 0.f;
  for (int j = threadIdx.x * 8; j < vocab; j += 256 * 8) {
    float v[8];
    Vec8<T>::load(row + j, v);
    float mx = v[0];
#pragma unroll
    for (int i = 1; i < 8; ++i) mx = fmaxf(mx, v[i]);
    const float mn = fmaxf(m, mx);
    float acc = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) acc += __expf(v[i] - mn);
    s = s * __expf(m - mn) + acc;
    m = mn;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, s, o);
    ms_merge(m, s, m2, s2);
  }
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { sm_m[w] = m; sm_s[w] = s; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < 8; ++i) ms_merge(m, s, sm_m[i], sm_s[i]);
    const float lse = m + logf(s);
    row_lse[r] = lse;
    const float tgt = to_f32(row[labels[r]]);
    atomicAdd(loss_acc, coef * (lse - tgt));
  }
}
// d logits = upstream * coef * (softmax - onehot), written in place over the logits buffer
template <typename T>
__global__ void __launch_bounds__(256) ce_bwd_kernel(T* __restrict__ logits, const long long* __restrict__ labels, int vocab, float coef,
                                                     const float* __restrict__ row_lse, const float* __restrict__ upstream) {
  const int r = blockIdx.x;
  T* row = logits + (long long)r * vocab;
  const float lse = row_lse[r];
  const float gsc = coef * __ldg(upstream);
  const int lab = (int)labels[r];
  for (int j = threadIdx.x * 8; j < vocab; j += 256 * 8) {
    float v[8];
    Vec8<T>::load(row + j, v);
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = gsc * (__expf(v[i] - lse) - ((j + i) == lab ? 1.f : 0.f));
    Vec8<T>::store(row + j, v);
  }
}

// Head split + rotary + q scale as a streaming pass over the plain to_qkv output (attention.py:63-69): qkv [rows, 3*h*dh] ->
// q,k,v [b,h,n,dh].  Thread = 8 channels; the 8 lanes of a head read one 128-byte cos / sin table row and write one 128-byte
// q/k/v row, so every access is a full line.  (Measured faster than doing the same in the tcgen05 epilogue, where a thread
// owns a token row and its table loads are 32 different lines per instruction; profiles/r01_summary.md.)
template <typename T>
__global__ void __launch_bounds__(256) qkv_rotary_kernel(const T* __restrict__ qkv, T* __restrict__ q, T* __restrict__ k, T* __restrict__ v,
                                                         const float* __restrict__ cos_t, const float* __restrict__ sin_t, int rows, int seq_n,
                                                         int heads, int dh, int pos_offset, float q_scale, int n_alloc) {
  pdl_launch();
  pdl_wait();
  const int inner = heads * dh;
  const int m = blockIdx.x;                                      // token row (block-uniform: its b / p split costs nothing)
  const int c = (blockIdx.y * 256 + threadIdx.x) * 8;            // column in [0, 3*inner)
  if (c >= 3 * inner) return;
  const int which = c >= 2 * inner ? 2 : (c >= inner ? 1 : 0);
  const int rem = c - which * inner;
  const int head = rem / dh, d = rem - head * dh;
  const int b = m / seq_n, p = m - b * seq_n;
  float x[8];
  Vec8<T>::load(qkv + (long long)m * (3 * inner) + c, x);
  if (cos_t) {
    const int ti = (p + pos_offset) * (dh >> 1) + (d >> 1);
    const float4 cc = __ldg(reinterpret_cast<const float4*>(cos_t + ti));
    const float4 ss = __ldg(reinterpret_cast<const float4*>(sin_t + ti));
    const float cv[4] = {cc.x, cc.y, cc.z, cc.w}, sv[4] = {ss.x, ss.y, ss.z, ss.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float x0 = x[2 * i], x1 = x[2 * i + 1];
      x[2 * i] = x0 * cv[i] + (-x1) * sv[i];
      x[2 * i + 1] = x1 * cv[i] + x0 * sv[i];
    }
  }
  if (which == 0) {
#pragma unroll
    for (int i = 0; i < 8; ++i) x[i] *= q_scale;
  }
  T* base = which == 0 ? q : (which == 1 ? k : v);
  T* dst = base + (((long long)b * heads + head) * n_alloc + p) * dh + d;
  Vec8<T>::store(dst, x);
  if (p == seq_n - 1 && n_alloc > seq_n) {      // zero token(s) behind the sequence (gathered axial layout)
#pragma unroll
    for (int i = 0; i < 8; ++i) x[i] = 0.f;
    for (int r = 1; r <= n_alloc - seq_n; ++r) Vec8<T>::store(dst + (long long)r * dh, x);
  }
}

constexpr int CS_ROWS = 512;
template <typename T>
__global__ void __launch_bounds__(256) colsum_kernel(const T* __restrict__ x, int rows, int cols, float* __restrict__ out) {
  __shared__ float red[8][64];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int c = (blockIdx.x * 32 + tx) * 2;
  const int r0 = blockIdx.y * CS_ROWS;
  const int r1 = min(rows, r0 + CS_ROWS);
  float a0 = 0.f, a1 = 0.f;
  if (c < cols) {
    for (int r = r0 + ty; r < r1; r += 8) {
      const float2 v = load2<T>(x + (long long)r * cols + c);
      a0 += v.x; a1 += v.y;
    }
  }
  red[ty][tx * 2] = a0; red[ty][tx * 2 + 1] = a1;
  __syncthreads();
  if (ty == 0 && c < cols) {
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) { s0 += red[i][tx * 2]; s1 += red[i][tx * 2 + 1]; }
    atomicAdd(out + c, s0);
    atomicAdd(out + c + 1, s1);
  }
}

__global__ void cast_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, long long count) {
  pdl_launch();
  pdl_wait();
  const long long stride = (long long)gridDim.x * blockDim.x * 4;
  for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < count; i += stride) {
    if (i + 3 < count) {
      const float4 v = *reinterpret_cast<const float4*>(src + i);
      *reinterpret_cast<__nv_bfloat162*>(dst + i) = __floats2bfloat162_rn(v.x, v.y);
      *reinterpret_cast<__nv_bfloat162*>(dst + i + 2) = __floats2bfloat162_rn(v.z, v.w);
    } else {
      for (long long j = i; j < count; ++j) dst[j] = __float2bfloat16_rn(src[j]);
    }
  }
}

__global__ void axpby_kernel(const float* __restrict__ a, const float* __restrict__ b, float alpha, float* __restrict__ y,
                             long long count) {
  const long long stride = (long long)gridDim.x * blockDim.x * 4;
  for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < count; i += stride) {
    if (i + 3 < count) {
      const float4 u = *reinterpret_cast<const float4*>(a + i);
      const float4 v = *reinterpret_cast<const float4*>(b + i);
      *reinterpret_cast<float4*>(y + i) = make_float4(u.x + alpha * v.x, u.y + alpha * v.y, u.z + alpha * v.z, u.w + alpha * v.w);
    } else {
      for (long long j = i; j < count; ++j) y[j] = a[j] + alpha * b[j];
    }
  }
}

// ---- optimizer step (train_dalle.py:617-619) over flat buffers ----------------------------------------------------------
__global__ void __launch_bounds__(256) sumsq_kernel(const float* __restrict__ x, long long count, float* __restrict__ out) {
  float acc = 0.f;
  const long long stride = (long long)gridDim.x * blockDim.x * 4;
  for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < count; i += stride) {
    if (i + 3 < count) {
      const float4 v = *reinterpret_cast<const float4*>(x + i);
      acc += (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
    } else {
      for (long long j = i; j < count; ++j) acc += x[j] * x[j];
    }
  }
  acc = warp_sum(acc);
  __shared__ float red[8];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += red[i];
    atomicAdd(out, t);
  }
}
__device__ __forceinline__ void adam_one(float& p, float g, float& m, float& v, float coef, float wd, float b1, float b2, float step_size,
                                         float inv_sqrt_bc2, float eps) {
  g = g * coef + wd * p;
  m = m + (1.0f - b1) * (g - m);                       // exp_avg.lerp_(grad, 1 - beta1)
  v = b2 * v + (1.0f - b2) * g * g;
  p -= step_size * m / (sqrtf(v) * inv_sqrt_bc2 + eps);
}
__global__ void __launch_bounds__(256) adam_kernel(db200_adam_params P, float step_size, float inv_sqrt_bc2) {
  float coef = 1.0f;
  if (P.max_norm > 0.f) {
    const float c = P.max_norm / (sqrtf(__ldg(P.gnorm_sq)) + 1e-6f);
    coef = c < 1.0f ? c : 1.0f;
  }
  const long long stride = (long long)gridDim.x * blockDim.x * 4;
  for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < P.count; i += stride) {
    if (i + 3 < P.count) {
      float4 p = *reinterpret_cast<float4*>(P.p + i), m = *reinterpret_cast<float4*>(P.m + i), v = *reinterpret_cast<float4*>(P.v + i);
      const float4 g = *reinterpret_cast<const float4*>(P.g + i);
      adam_one(p.x, g.x, m.x, v.x, coef, P.weight_decay, P.beta1, P.beta2, step_size, inv_sqrt_bc2, P.eps);
      adam_one(p.y, g.y, m.y, v.y, coef, P.weight_decay, P.beta1, P.beta2, step_size, inv_sqrt_bc2, P.eps);
      adam_one(p.z, g.z, m.z, v.z, coef, P.weight_decay, P.beta1, P.beta2, step_size, inv_sqrt_bc2, P.eps);
      adam_one(p.w, g.w, m.w, v.w, coef, P.weight_decay, P.beta1, P.beta2, step_size, inv_sqrt_bc2, P.eps);
      *reinterpret_cast<float4*>(P.p + i) = p; *reinterpret_cast<float4*>(P.m + i) = m; *reinterpret_cast<float4*>(P.v + i) = v;
    } else {
      for (long long j = i; j < P.count; ++j) adam_one(P.p[j], P.g[j], P.m[j], P.v[j], coef, P.weight_decay, P.beta1, P.beta2, step_size, inv_sqrt_bc2, P.eps);
    }
  }
}

// token embedding gather / scatter-add: one warp per token row, 16 bytes per lane and step
__global__ void __launch_bounds__(256) embed_fwd_kernel(const long long* __restrict__ ids, const float* __restrict__ w, float* __restrict__ out,
                                                        int rows, int seg_len, int n, int seg_off, int d, int vocab) {
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (r >= rows) return;
  const int b = r / seg_len, l = r - b * seg_len;
  long long id = ids[r];
  if (id < 0 || id >= vocab) id = 0;                       // validated on the host side of the module; never index out of range
  const float* src = w + id * d;
  float* dst = out + ((long long)b * n + seg_off + l) * d;
  for (int c = lane * 4; c < d; c += 128) *reinterpret_cast<float4*>(dst + c) = __ldg(reinterpret_cast<const float4*>(src + c));
}
__global__ void __launch_bounds__(256) embed_bwd_kernel(const long long* __restrict__ ids, const float* __restrict__ g, float* __restrict__ dw,
                                                        int rows, int seg_len, int n, int seg_off, int d, int vocab) {
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (r >= rows) return;
  const int b = r / seg_len, l = r - b * seg_len;
  const long long id = ids[r];
  if (id < 0 || id >= vocab) return;
  const float* src = g + ((long long)b * n + seg_off + l) * d;
  float* dst = dw + id * d;
  for (int c = lane * 4; c < d; c += 128) {
    const float4 v = *reinterpret_cast<const float4*>(src + c);
    atomicAdd(dst + c, v.x); atomicAdd(dst + c + 1, v.y); atomicAdd(dst + c + 2, v.z); atomicAdd(dst + c + 3, v.w);
  }
}

}  // namespace

int sumsq_launch(const float* x, int64_t count, float* out, cudaStream_t st) {
  if (count == 0) return DB200_OK;
  int64_t blocks = ceil_div64(count, 256 * 4 * 4);
  if (blocks > sm_count() * 8) blocks = sm_count() * 8;
  if (blocks < 1) blocks = 1;
  sumsq_kernel<<<(int)blocks, 256, 0, st>>>(x, count, out);
  DB200_LAUNCH_OK("sumsq_kernel");
  return DB200_OK;
}
int adam_launch(const db200_adam_params& P, cudaStream_t st) {
  if (P.count == 0) return DB200_OK;
  const double bc1 = 1.0 - pow((double)P.beta1, (double)P.step), bc2 = 1.0 - pow((double)P.beta2, (double)P.step);
  int64_t blocks = ceil_div64(P.count, 256 * 4 * 2);
  if (blocks > sm_count() * 8) blocks = sm_count() * 8;
  if (blocks < 1) blocks = 1;
  adam_kernel<<<(int)blocks, 256, 0, st>>>(P, (float)(P.lr / bc1), (float)(1.0 / sqrt(bc2)));
  DB200_LAUNCH_OK("adam_kernel");
  return DB200_OK;
}

int embed_launch(bool bwd, const long long* ids, const float* a, float* o, int batch, int seg_len, int n, int seg_off, int d, int vocab,
                 cudaStream_t st) {
  const int rows = batch * seg_len;
  if (rows == 0) return DB200_OK;
  if (bwd) embed_bwd_kernel<<<ceil_div(rows, 8), 256, 0, st>>>(ids, a, o, rows, seg_len, n, seg_off, d, vocab);
  else embed_fwd_kernel<<<ceil_div(rows, 8), 256, 0, st>>>(ids, a, o, rows, seg_len, n, seg_off, d, vocab);
  DB200_LAUNCH_OK("embed_kernel");
  return DB200_OK;
}

int ln_shift_fwd_launch(const db200_ln_shift_fwd_params& P, cudaStream_t st) {
  const int rows = P.batch * P.n;
  if (rows == 0) return DB200_OK;
  const int wgrid = ceil_div(rows, WR_WARPS);
#define DB200_LN_FWD_WARP(NCH)                                                                                              \
  do {                                                                                                                      \
    if (P.out_dtype == DB200_F32) DB200_CUDA_OK(launch_pdl(ln_shift_fwd_warp_kernel<float, NCH>, dim3(wgrid), dim3(WR_WARPS * 32), 0, st, P)); \
    else DB200_CUDA_OK(launch_pdl(ln_shift_fwd_warp_kernel<__nv_bfloat16, NCH>, dim3(wgrid), dim3(WR_WARPS * 32), 0, st, P));              \
    DB200_LAUNCH_OK("ln_shift_fwd_warp_kernel");                                                                           \
    return DB200_OK;                                                                                                        \
  } while (0)
  if (P.d == 256) DB200_LN_FWD_WARP(2);
  if (P.d == 512) DB200_LN_FWD_WARP(4);
  if (P.d == 1024) DB200_LN_FWD_WARP(8);
  if (P.d == 2048) DB200_LN_FWD_WARP(16);
#undef DB200_LN_FWD_WARP
  const size_t smem = (size_t)P.d * sizeof(float);
  if (P.out_dtype == DB200_F32) ln_shift_fwd_kernel<float><<<rows, LN_THREADS, smem, st>>>(P);
  else ln_shift_fwd_kernel<__nv_bfloat16><<<rows, LN_THREADS, smem, st>>>(P);
  DB200_LAUNCH_OK("ln_shift_fwd_kernel");
  return DB200_OK;
}

int ln_shift_bwd_launch(const db200_ln_shift_bwd_params& P, cudaStream_t st) {
  const int rows = P.batch * P.n;
  if (rows == 0) return DB200_OK;
  const bool al16 = ((reinterpret_cast<uintptr_t>(P.d_out) | reinterpret_cast<uintptr_t>(P.x) | reinterpret_cast<uintptr_t>(P.dres)) & 15) == 0;
  static const bool no_tma = [] { const char* v = getenv("DALLE_B200_LN_BWD"); return v && !strcmp(v, "regs"); }();
  if (P.up_dy && !(P.d == 1024 && al16)) return set_error(DB200_ERR_UNSUPPORTED, "ln_shift_bwd: fused upstream adjoint needs d = 1024 and aligned tensors");
  if (P.d == 1024 && al16 && (!no_tma || P.up_dy)) {
    const int want = ceil_div(rows, LT_R);
    const int grid = want < sm_count() ? want : sm_count();
    if (P.dout_dtype == DB200_F32) {
      static std::atomic<bool> attr{false};   // idempotent set-up; atomic because forward and autograd threads both launch
      if (!attr.load(std::memory_order_acquire)) { DB200_CUDA_OK(cudaFuncSetAttribute(ln_shift_bwd_tma_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, LnTmaSmem<float>::TOTAL)); attr.store(true, std::memory_order_release); }
      DB200_CUDA_OK(launch_pdl(ln_shift_bwd_tma_kernel<float>, dim3(grid), dim3(LT_THREADS), LnTmaSmem<float>::TOTAL, st, P));
    } else {
      static std::atomic<bool> attr{false};   // idempotent set-up; atomic because forward and autograd threads both launch
      if (!attr.load(std::memory_order_acquire)) { DB200_CUDA_OK(cudaFuncSetAttribute(ln_shift_bwd_tma_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, LnTmaSmem<__nv_bfloat16>::TOTAL)); attr.store(true, std::memory_order_release); }
      DB200_CUDA_OK(launch_pdl(ln_shift_bwd_tma_kernel<__nv_bfloat16>, dim3(grid), dim3(LT_THREADS), LnTmaSmem<__nv_bfloat16>::TOTAL, st, P));
    }
    DB200_LAUNCH_OK("ln_shift_bwd_tma_kernel");
    return DB200_OK;
  }
  if (P.d == 256 || P.d == 512 || P.d == 1024) {
    const int want = ceil_div(rows, WR_WARPS);
    const int wgrid = want < sm_count() * 3 ? want : sm_count() * 3;
    const size_t wsmem = (size_t)2 * P.d * sizeof(float);
#define DB200_LN_BWD_DX(NCH)                                                                                                \
  do {                                                                                                                      \
    if (P.dout_dtype == DB200_F32) ln_shift_bwd_dx_kernel<float, NCH><<<wgrid, WR_WARPS * 32, wsmem, st>>>(P);             \
    else ln_shift_bwd_dx_kernel<__nv_bfloat16, NCH><<<wgrid, WR_WARPS * 32, wsmem, st>>>(P);                               \
  } while (0)
    if (P.d == 256) DB200_LN_BWD_DX(2);
    else if (P.d == 512) DB200_LN_BWD_DX(4);
    else DB200_LN_BWD_DX(8);
#undef DB200_LN_BWD_DX
    DB200_LAUNCH_OK("ln_shift_bwd_dx_kernel");
    return DB200_OK;
  }
  const size_t smem = (size_t)4 * P.d * sizeof(float);
  const int grid = rows < sm_count() * 8 ? rows : sm_count() * 8;
  if (P.dout_dtype == DB200_F32) ln_shift_bwd_kernel<float><<<grid, LN_THREADS, smem, st>>>(P);
  else ln_shift_bwd_kernel<__nv_bfloat16><<<grid, LN_THREADS, smem, st>>>(P);
  DB200_LAUNCH_OK("ln_shift_bwd_kernel");
  return DB200_OK;
}

// Rows per CTA for the slab-streaming kernels: the grid must be whole waves of resident CTAs (148 SMs x `resident`), otherwise
// the last partial wave runs at a fraction of the HBM bandwidth (measured: 640 CTAs on 592 slots = 2 waves for 1.08 waves of
// work).  One wave, chunk rounded up to `quantum` rows.
static int balanced_rows_per_block(int rows, int col_blocks, int resident, int quantum) {
  const int slots = sm_count() * resident / (col_blocks > 0 ? col_blocks : 1);
  if (slots <= 0) return rows;
  int rpb = ceil_div(rows, slots);          // one wave; small inputs keep at least 32 rows per CTA (fewer CTAs than slots)
  if (rpb < 32) rpb = 32;
  rpb = ceil_div(rpb, quantum) * quantum;
  return rpb;
}

int scale_bwd_launch(const db200_scale_bwd_params& P, cudaStream_t st) {
  if (P.rows == 0) return DB200_OK;
  const size_t smem = (size_t)2 * P.d * sizeof(float);
  if ((P.d & 3) == 0) {
    const int cb = ceil_div(P.d, 1024);
    const int rpb = balanced_rows_per_block(P.rows, cb, 2, 8);
    dim3 sgrid(cb, ceil_div(P.rows, rpb));
    if (P.dtype == DB200_F32) DB200_CUDA_OK(launch_pdl(scale_bwd_slab_kernel<float>, sgrid, dim3(256), 0, st, P, rpb));
    else DB200_CUDA_OK(launch_pdl(scale_bwd_slab_kernel<__nv_bfloat16>, sgrid, dim3(256), 0, st, P, rpb));
    DB200_LAUNCH_OK("scale_bwd_slab_kernel");
    return DB200_OK;
  }
  const int grid = P.rows < sm_count() * 4 ? P.rows : sm_count() * 4;
  if (P.dtype == DB200_F32) scale_bwd_kernel<float><<<grid, 256, smem, st>>>(P);
  else scale_bwd_kernel<__nv_bfloat16><<<grid, 256, smem, st>>>(P);
  DB200_LAUNCH_OK("scale_bwd_kernel");
  return DB200_OK;
}

int geglu_bwd_launch(const void* dh, const void* u, void* du, float* dbias, int dtype, int rows, int hidden, cudaStream_t st) {
  if (rows == 0) return DB200_OK;
  const int cb = ceil_div(hidden, 2048);
  const int rpb = balanced_rows_per_block(rows, cb, 4, 4);
  dim3 grid(cb, ceil_div(rows, rpb));
  if (dtype == DB200_F32)
    DB200_CUDA_OK(launch_pdl(geglu_bwd_kernel<float>, grid, dim3(256), 0, st, reinterpret_cast<const float*>(dh), reinterpret_cast<const float*>(u),
                             reinterpret_cast<float*>(du), dbias, rows, hidden, rpb));
  else
    DB200_CUDA_OK(launch_pdl(geglu_bwd_kernel<__nv_bfloat16>, grid, dim3(256), 0, st, reinterpret_cast<const __nv_bfloat16*>(dh),
                             reinterpret_cast<const __nv_bfloat16*>(u), reinterpret_cast<__nv_bfloat16*>(du), dbias, rows, hidden, rpb));
  DB200_LAUNCH_OK("geglu_bwd_kernel");
  return DB200_OK;
}

int ce_fwd_launch(const void* logits, int dtype, int rows, int vocab, const long long* labels, float coef, float* row_lse, float* loss_acc,
                  cudaStream_t st) {
  if (rows == 0) return DB200_OK;
  if (dtype == DB200_F32) ce_fwd_kernel<float><<<rows, 256, 0, st>>>(reinterpret_cast<const float*>(logits), labels, vocab, coef, row_lse, loss_acc);
  else ce_fwd_kernel<__nv_bfloat16><<<rows, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(logits), labels, vocab, coef, row_lse, loss_acc);
  DB200_LAUNCH_OK("ce_fwd_kernel");
  return DB200_OK;
}
int ce_bwd_launch(void* logits, int dtype, int rows, int vocab, const long long* labels, float coef, const float* row_lse, const float* upstream,
                  cudaStream_t st) {
  if (rows == 0) return DB200_OK;
  if (dtype == DB200_F32) ce_bwd_kernel<float><<<rows, 256, 0, st>>>(reinterpret_cast<float*>(logits), labels, vocab, coef, row_lse, upstream);
  else ce_bwd_kernel<__nv_bfloat16><<<rows, 256, 0, st>>>(reinterpret_cast<__nv_bfloat16*>(logits), labels, vocab, coef, row_lse, upstream);
  DB200_LAUNCH_OK("ce_bwd_kernel");
  return DB200_OK;
}

int qkv_rotary_launch(const void* qkv, void* q, void* k, void* v, const float* cos_t, const float* sin_t, int dtype, int rows, int seq_n, int heads,
                      int dh, int pos_offset, float q_scale, int n_alloc, cudaStream_t st) {
  if (rows == 0) return DB200_OK;
  const dim3 grid(rows, ceil_div(3 * heads * dh / 8, 256));
  if (dtype == DB200_F32)
    DB200_CUDA_OK(launch_pdl(qkv_rotary_kernel<float>, grid, dim3(256), 0, st, reinterpret_cast<const float*>(qkv), reinterpret_cast<float*>(q),
                             reinterpret_cast<float*>(k), reinterpret_cast<float*>(v), cos_t, sin_t, rows, seq_n, heads, dh, pos_offset, q_scale, n_alloc));
  else
    DB200_CUDA_OK(launch_pdl(qkv_rotary_kernel<__nv_bfloat16>, grid, dim3(256), 0, st, reinterpret_cast<const __nv_bfloat16*>(qkv),
                             reinterpret_cast<__nv_bfloat16*>(q), reinterpret_cast<__nv_bfloat16*>(k), reinterpret_cast<__nv_bfloat16*>(v), cos_t, sin_t,
                             rows, seq_n, heads, dh, pos_offset, q_scale, n_alloc));
  DB200_LAUNCH_OK("qkv_rotary_kernel");
  return DB200_OK;
}

int colsum_launch(const void* x, int dtype, int rows, int cols, float* out, cudaStream_t st) {
  if (rows == 0 || cols == 0) return DB200_OK;
  dim3 grid(ceil_div(cols, 64), ceil_div(rows, CS_ROWS));
  if (dtype == DB200_F32) colsum_kernel<float><<<grid, 256, 0, st>>>(reinterpret_cast<const float*>(x), rows, cols, out);
  else colsum_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(x), rows, cols, out);
  DB200_LAUNCH_OK("colsum_kernel");
  return DB200_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// fp32 GEMMs on the bf16 tensor cores (parity mode "bf16x6"): x = x0 + x1 + x2 with x0 = bf16(x), x1 = bf16(x - x0),
// x2 = bf16(x - x0 - x1) carries 24 mantissa bits; A B^T = sum over (i,j) in {(0,0),(0,1),(1,0),(1,1),(0,2),(2,0)} of Ai Bj^T up to
// terms of relative size 2^-24.  The six products are ONE tcgen05 GEMM over a K axis six times as long: this kernel writes the
// pieces side by side along K in the order the operand needs (`pat` = piece index of each of the six K blocks), so
// gemm_tcgen05_kernel, its operand-major modes and its fp32 accumulator in tensor memory are used unchanged.
//   concat_rows == 0: src [rows, cols] -> dst [rows, 6*cols]  (K contiguous: K-major operand)
//   concat_rows == 1: src [rows, cols] -> dst [6*rows, cols]  (K = the row index: MN-major operand)
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) split_bf16x3_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, long long rows, int cols,
                                                           int concat_rows, int pat) {
  pdl_launch();
  pdl_wait();
  const long long total = rows * (long long)(cols >> 1);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / (cols >> 1);
    const int c = static_cast<int>(i - r * (cols >> 1)) * 2;
    const float2 x = *reinterpret_cast<const float2*>(src + r * cols + c);
    __nv_bfloat162 pc[3];
    float2 rem = x;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      pc[k] = __floats2bfloat162_rn(rem.x, rem.y);
      const float2 back = __bfloat1622float2(pc[k]);
      rem.x -= back.x; rem.y -= back.y;                     // exact: the difference of x and its bf16 rounding is representable
    }
#pragma unroll
    for (int blk = 0; blk < 6; ++blk) {
      const int which = (pat >> (4 * blk)) & 0xf;
      const long long off = concat_rows ? ((long long)blk * rows + r) * cols + c : r * (6LL * cols) + (long long)blk * cols + c;
      *reinterpret_cast<__nv_bfloat162*>(dst + off) = pc[which];
    }
  }
}

// out = resid + sign * scale (.) y      (fp32; the LayerScale + residual step of EPI_RESID as a streaming pass, parity mode)
template <typename T>
__global__ void __launch_bounds__(256) resid_scale_kernel(const T* __restrict__ y, const float* __restrict__ resid, const float* __restrict__ scale,
                                                          float sign, float* __restrict__ out, long long rows, int d) {
  pdl_launch();
  pdl_wait();
  const long long total = rows * (long long)(d >> 1);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / (d >> 1);
    const int c = static_cast<int>(i - r * (d >> 1)) * 2;
    const float2 v = load2<T>(y + r * d + c);
    float s0 = sign, s1 = sign;
    if (scale) { s0 *= scale[c]; s1 *= scale[c + 1]; }
    float2 o = make_float2(s0 * v.x, s1 * v.y);
    if (resid) { const float2 rr = *reinterpret_cast<const float2*>(resid + r * d + c); o.x += rr.x; o.y += rr.y; }
    *reinterpret_cast<float2*>(out + r * d + c) = o;
  }
}

// h = a * gelu_erf(g) with u = [a | g] [rows, 2*hidden]   (fp32; transformer.py:106-109, parity mode)
__global__ void __launch_bounds__(256) geglu_fwd_kernel(const float* __restrict__ u, float* __restrict__ hout, long long rows, int hidden) {
  pdl_launch();
  pdl_wait();
  const long long total = rows * (long long)hidden;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / hidden;
    const int j = static_cast<int>(i - r * hidden);
    const float a = u[r * (2LL * hidden) + j], g = u[r * (2LL * hidden) + hidden + j];
    hout[i] = a * gelu_erf(g);
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Dropout (attention.py:53-56 after to_out, transformer.py:117 after GEGLU) with a counter-based generator: element i keeps
// its value iff word (i & 3) of Philox4x32-10(key = seed, counter = offset + i / 4) is below the keep threshold, and is scaled
// by 1 / (1 - p).  The mask is a pure function of (seed, offset, i): the backward pass and the reversible executor's
// recomputation (reference Deterministic.record_rng / set_rng, reversible.py:20-50) replay it by passing the same pair.
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    const uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0; key.y += W1;
  }
  return ctr;
}

template <typename T>
__global__ void __launch_bounds__(256) dropout_kernel(const T* __restrict__ x, T* __restrict__ y, long long count, float p, float inv_keep,
                                                      unsigned long long seed, unsigned long long offset) {
  pdl_launch();
  pdl_wait();
  const uint32_t thresh = p <= 0.f ? 0xffffffffu : static_cast<uint32_t>(fminf((1.0f - p) * 4294967296.0f, 4294967295.0f));
  const uint2 key = make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
  const long long groups = (count + 3) >> 2;
  for (long long gidx = (long long)blockIdx.x * blockDim.x + threadIdx.x; gidx < groups; gidx += (long long)gridDim.x * blockDim.x) {
    const unsigned long long c = offset + static_cast<unsigned long long>(gidx);
    const uint4 r = philox4x32_10(make_uint4(static_cast<uint32_t>(c), static_cast<uint32_t>(c >> 32), 0u, 0u), key);
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
    const long long i0 = gidx << 2;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (i0 + j < count) {
        const float v = to_f32(x[i0 + j]);
        y[i0 + j] = from_f32<T>(w[j] <= thresh && p < 1.f ? v * inv_keep : 0.f);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Decoding: top-k filtering + Gumbel-max sampling of one token per row in ONE launch (dalle_pytorch.py:43-58, 533-539:
// top_k(logits, thres) keeps the k = max(int((1 - thres) * V), 1) largest logits, gumbel_sample draws
// argmax(logits / temperature + g), g = -log(-log(u))).  One CTA per row: the row is converted to order-preserving integer keys
// in shared memory, the k-th largest key is found by a 4-pass radix select (8 bits per pass, shared-memory histogram), then the
// block takes the arg-max of logit / T + g over the keys at or above it.  g comes from Philox4x32-10(seed, offset + element / 4)
// or, for tests, from an explicit [rows, V] tensor.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int SAMPLE_THREADS = 512;
__device__ __forceinline__ uint32_t float_key(float v) {            // ascending key order == ascending float order
  const uint32_t b = __float_as_uint(v);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

// logit i of the sampled row: the row itself, or (guided) null + (cond - null) * s evaluated as torch evaluates
// `null + (cond - null) * cond_scale` on tensors of dtype T -- three separately rounded operations in fp32 (no contraction), each
// result rounded to T -- so that the guided row equals torch's guided logits bit for bit
template <typename T>
struct PlainRow {
  const T* p;
  __device__ __forceinline__ float operator()(int i) const { return to_f32(p[i]); }
};
template <typename T>
struct GuidedRow {
  const T* cond; const T* null_; float s;
  __device__ __forceinline__ float operator()(int i) const {
    const float c = to_f32(cond[i]), u = to_f32(null_[i]);
    const float d = to_f32(from_f32<T>(__fsub_rn(c, u)));
    const float m = to_f32(from_f32<T>(__fmul_rn(d, s)));
    return to_f32(from_f32<T>(__fadd_rn(u, m)));
  }
};

template <typename Row>
__device__ __forceinline__ void sample_topk_gumbel_row(const Row lrow, int row, int V, int k, float inv_temp, const float* __restrict__ gumbel,
                                                       unsigned long long seed, unsigned long long offset, long long* __restrict__ out) {
  extern __shared__ uint32_t keys[];                                  // [V]
  __shared__ uint32_t hist[256];
  __shared__ uint32_t s_prefix, s_remaining;
  __shared__ float s_val[SAMPLE_THREADS / 32];
  __shared__ int s_idx[SAMPLE_THREADS / 32];
  const int tid = threadIdx.x;
  for (int i = tid; i < V; i += SAMPLE_THREADS) keys[i] = float_key(lrow(i));
  if (tid == 0) { s_prefix = 0u; s_remaining = static_cast<uint32_t>(k); }
  __syncthreads();
  uint32_t mask = 0u;
  for (int pass = 3; pass >= 0; --pass) {
    const int shift = pass * 8;
    if (tid < 256) hist[tid] = 0u;
    __syncthreads();
    const uint32_t prefix = s_prefix;
    for (int i = tid; i < V; i += SAMPLE_THREADS) {
      const uint32_t key = keys[i];
      if ((key & mask) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1u);
    }
    __syncthreads();
    if (tid == 0) {                                                   // walk the bins from the top: which digit holds the k-th largest
      uint32_t cum = 0u, rem = s_remaining;
      int b = 255;
      for (; b > 0; --b) {
        if (cum + hist[b] >= rem) break;
        cum += hist[b];
      }
      s_remaining = rem - cum;
      s_prefix = prefix | (static_cast<uint32_t>(b) << shift);
    }
    mask |= 0xffu << shift;
    __syncthreads();
  }
  const uint32_t kth = s_prefix;                                      // key of the k-th largest logit
  const uint2 pkey = make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
  float best = -INFINITY;
  int best_i = 0x7fffffff;
  for (int i = tid; i < V; i += SAMPLE_THREADS) {
    if (keys[i] < kth) continue;
    float g;
    if (gumbel) g = gumbel[(long long)row * V + i];
    else {
      const unsigned long long e = (unsigned long long)row * V + i, c = offset + (e >> 2);
      const uint4 r = philox4x32_10(make_uint4(static_cast<uint32_t>(c), static_cast<uint32_t>(c >> 32), 0u, 0u), pkey);
      const uint32_t w = (e & 3) == 0 ? r.x : (e & 3) == 1 ? r.y : (e & 3) == 2 ? r.z : r.w;
      const float u = (static_cast<float>(w >> 8) + 0.5f) * (1.0f / 16777216.0f);        // (0, 1)
      g = -logf(-logf(u + 1e-20f) + 1e-20f);                         // dalle_pytorch.py:50-52
    }
    const float v = lrow(i) * inv_temp + g;
    if (v > best || (v == best && i < best_i)) { best = v; best_i = i; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
    if (ov > best || (ov == best && oi < best_i)) { best = ov; best_i = oi; }
  }
  if ((tid & 31) == 0) { s_val[tid >> 5] = best; s_idx[tid >> 5] = best_i; }
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < SAMPLE_THREADS / 32; ++w)
      if (s_val[w] > best || (s_val[w] == best && s_idx[w] < best_i)) { best = s_val[w]; best_i = s_idx[w]; }
    out[row] = best_i;
  }
}

template <typename T>
__global__ void __launch_bounds__(SAMPLE_THREADS) sample_topk_gumbel_kernel(const T* __restrict__ logits, int V, long long ld, int k, float inv_temp,
                                                                           const float* __restrict__ gumbel, unsigned long long seed,
                                                                           unsigned long long offset, long long* __restrict__ out) {
  const int row = blockIdx.x;
  sample_topk_gumbel_row(PlainRow<T>{logits + (long long)row * ld}, row, V, k, inv_temp, gumbel, seed, offset, out);
}

// classifier-free guidance: row r of the guided logits is formed from cond row r and null row r on the fly (never written); the
// Philox counters are those of a [rows, V] guided logits tensor passed to sample_topk_gumbel_kernel
template <typename T>
__global__ void __launch_bounds__(SAMPLE_THREADS) sample_guided_topk_gumbel_kernel(const T* __restrict__ cond, const T* __restrict__ null_, long long ld,
                                                                                  float cond_scale, int V, int k, float inv_temp,
                                                                                  const float* __restrict__ gumbel, unsigned long long seed,
                                                                                  unsigned long long offset, long long* __restrict__ out) {
  const int row = blockIdx.x;
  sample_topk_gumbel_row(GuidedRow<T>{cond + (long long)row * ld, null_ + (long long)row * ld, cond_scale}, row, V, k, inv_temp, gumbel, seed,
                         offset, out);
}

int sample_topk_gumbel_launch(const void* logits, int dtype, int rows, int vocab, long long ld, int k, float temperature, const float* gumbel,
                              unsigned long long seed, unsigned long long offset, long long* out, cudaStream_t st) {
  if (rows == 0) return DB200_OK;
  const size_t smem = (size_t)vocab * 4;
  static std::atomic<bool> attr_done{false};
  if (!attr_done.load(std::memory_order_acquire)) {
    DB200_CUDA_OK(cudaFuncSetAttribute(sample_topk_gumbel_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    DB200_CUDA_OK(cudaFuncSetAttribute(sample_topk_gumbel_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr_done.store(true, std::memory_order_release);
  }
  const float inv_temp = 1.0f / temperature;
  if (dtype == DB200_F32)
    sample_topk_gumbel_kernel<float><<<rows, SAMPLE_THREADS, smem, st>>>(reinterpret_cast<const float*>(logits), vocab, ld, k, inv_temp, gumbel, seed, offset, out);
  else
    sample_topk_gumbel_kernel<__nv_bfloat16><<<rows, SAMPLE_THREADS, smem, st>>>(reinterpret_cast<const __nv_bfloat16*>(logits), vocab, ld, k, inv_temp, gumbel,
                                                                               seed, offset, out);
  DB200_LAUNCH_OK("sample_topk_gumbel_kernel");
  return DB200_OK;
}

int sample_guided_topk_gumbel_launch(const void* cond, const void* null_logits, int dtype, int rows, int vocab, long long ld, float cond_scale, int k,
                                     float temperature, const float* gumbel, unsigned long long seed, unsigned long long offset, long long* out,
                                     cudaStream_t st) {
  if (rows == 0) return DB200_OK;
  const size_t smem = (size_t)vocab * 4;
  static std::atomic<bool> attr_done{false};
  if (!attr_done.load(std::memory_order_acquire)) {
    DB200_CUDA_OK(cudaFuncSetAttribute(sample_guided_topk_gumbel_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    DB200_CUDA_OK(cudaFuncSetAttribute(sample_guided_topk_gumbel_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr_done.store(true, std::memory_order_release);
  }
  const float inv_temp = 1.0f / temperature;
  if (dtype == DB200_F32)
    sample_guided_topk_gumbel_kernel<float><<<rows, SAMPLE_THREADS, smem, st>>>(reinterpret_cast<const float*>(cond), reinterpret_cast<const float*>(null_logits),
                                                                                ld, cond_scale, vocab, k, inv_temp, gumbel, seed, offset, out);
  else
    sample_guided_topk_gumbel_kernel<__nv_bfloat16><<<rows, SAMPLE_THREADS, smem, st>>>(reinterpret_cast<const __nv_bfloat16*>(cond),
                                                                                        reinterpret_cast<const __nv_bfloat16*>(null_logits), ld, cond_scale,
                                                                                        vocab, k, inv_temp, gumbel, seed, offset, out);
  DB200_LAUNCH_OK("sample_guided_topk_gumbel_kernel");
  return DB200_OK;
}

static int grid_for(long long work) {
  long long blocks = (work + 255) / 256;
  const long long cap = (long long)sm_count() * 16;
  return static_cast<int>(blocks < 1 ? 1 : (blocks > cap ? cap : blocks));
}

int split_bf16x3_launch(const float* src, void* dst, int64_t rows, int cols, int concat_rows, int pat, cudaStream_t st) {
  if (rows == 0 || cols == 0) return DB200_OK;
  DB200_CUDA_OK(launch_pdl(split_bf16x3_kernel, dim3(grid_for(rows * (cols / 2))), dim3(256), 0, st, src, reinterpret_cast<__nv_bfloat16*>(dst),
                           (long long)rows, cols, concat_rows, pat));
  DB200_LAUNCH_OK("split_bf16x3_kernel");
  return DB200_OK;
}

int resid_scale_launch(const void* y, int dtype, const float* resid, const float* scale, float sign, float* out, int64_t rows, int d, cudaStream_t st) {
  if (rows == 0) return DB200_OK;
  if (dtype == DB200_F32)
    DB200_CUDA_OK(launch_pdl(resid_scale_kernel<float>, dim3(grid_for(rows * (d / 2))), dim3(256), 0, st, reinterpret_cast<const float*>(y), resid, scale,
                             sign, out, (long long)rows, d));
  else
    DB200_CUDA_OK(launch_pdl(resid_scale_kernel<__nv_bfloat16>, dim3(grid_for(rows * (d / 2))), dim3(256), 0, st,
                             reinterpret_cast<const __nv_bfloat16*>(y), resid, scale, sign, out, (long long)rows, d));
  DB200_LAUNCH_OK("resid_scale_kernel");
  return DB200_OK;
}

int geglu_fwd_launch(const float* u, float* h, int64_t rows, int hidden, cudaStream_t st) {
  if (rows == 0) return DB200_OK;
  DB200_CUDA_OK(launch_pdl(geglu_fwd_kernel, dim3(grid_for(rows * hidden)), dim3(256), 0, st, u, h, (long long)rows, hidden));
  DB200_LAUNCH_OK("geglu_fwd_kernel");
  return DB200_OK;
}

int dropout_launch(const void* x, void* y, int dtype, int64_t count, float p, unsigned long long seed, unsigned long long offset, cudaStream_t st) {
  if (count == 0) return DB200_OK;
  const float inv_keep = p < 1.f ? 1.0f / (1.0f - p) : 0.f;
  const int grid = grid_for((count + 3) / 4);
  if (dtype == DB200_F32)
    DB200_CUDA_OK(launch_pdl(dropout_kernel<float>, dim3(grid), dim3(256), 0, st, reinterpret_cast<const float*>(x), reinterpret_cast<float*>(y),
                             (long long)count, p, inv_keep, seed, offset));
  else
    DB200_CUDA_OK(launch_pdl(dropout_kernel<__nv_bfloat16>, dim3(grid), dim3(256), 0, st, reinterpret_cast<const __nv_bfloat16*>(x),
                             reinterpret_cast<__nv_bfloat16*>(y), (long long)count, p, inv_keep, seed, offset));
  DB200_LAUNCH_OK("dropout_kernel");
  return DB200_OK;
}

// mc_dst[i] += scale * src[i] in every GPU's replica (multimem.red through the NVLink multicast address)
__global__ void __launch_bounds__(256) mc_add_kernel(const float* __restrict__ src, float* mc_dst, long long count, float scale) {
  pdl_launch();
  pdl_wait();
  const long long groups = count >> 2;
  for (long long gidx = (long long)blockIdx.x * blockDim.x + threadIdx.x; gidx < groups; gidx += (long long)gridDim.x * blockDim.x) {
    const float4 v = *reinterpret_cast<const float4*>(src + 4 * gidx);
    asm volatile("multimem.red.relaxed.sys.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc_dst + 4 * gidx), "f"(v.x * scale), "f"(v.y * scale),
                 "f"(v.z * scale), "f"(v.w * scale)
                 : "memory");
  }
  if (blockIdx.x == 0 && threadIdx.x < (count & 3)) {
    const long long i = (groups << 2) + threadIdx.x;
    asm volatile("multimem.red.relaxed.sys.global.add.f32 [%0], %1;" ::"l"(mc_dst + i), "f"(src[i] * scale) : "memory");
  }
}

int mc_add_launch(const float* src, void* mc_dst, int64_t count, float scale, cudaStream_t st) {
  if (count == 0) return DB200_OK;
  DB200_CUDA_OK(launch_pdl(mc_add_kernel, dim3(grid_for((count + 3) / 4)), dim3(256), 0, st, src, reinterpret_cast<float*>(mc_dst), (long long)count,
                           scale));
  DB200_LAUNCH_OK("mc_add_kernel");
  return DB200_OK;
}

int cast_bf16_launch(const float* src, void* dst, int64_t count, cudaStream_t st) {
  if (count == 0) return DB200_OK;
  int64_t blocks = ceil_div64(count, 256 * 4);
  if (blocks > sm_count() * 16) blocks = sm_count() * 16;
  DB200_CUDA_OK(launch_pdl(cast_bf16_kernel, dim3((int)blocks), dim3(256), 0, st, src, reinterpret_cast<__nv_bfloat16*>(dst), (long long)count));
  DB200_LAUNCH_OK("cast_bf16_kernel");
  return DB200_OK;
}

int axpby_launch(const float* a, const float* b, float alpha, float* y, int64_t count, cudaStream_t st) {
  if (count == 0) return DB200_OK;
  int64_t blocks = ceil_div64(count, 256 * 4);
  if (blocks > sm_count() * 16) blocks = sm_count() * 16;
  axpby_kernel<<<(int)blocks, 256, 0, st>>>(a, b, alpha, y, count);
  DB200_LAUNCH_OK("axpby_kernel");
  return DB200_OK;
}

}  // namespace db200
