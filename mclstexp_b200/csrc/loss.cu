// Symmetric contrastive loss, forward + backward, for identity targets (reference
// model.py:242-247) and BLEEP soft targets (baselines/Bleep/models.py:34-43, :70-79 and
// cross_entropy :228-234), without ever holding a B x B matrix for more than one row block.
//
// With Lg = S I^T / T,  A = (I I^T + S S^T) * a   (a = 1/(2T) "div" or T/2 "mul"),
// Pt = softmax_row(A) (soft) or the identity (eye), rl/cl the row/column log-sum-exp of Lg,
// za the row log-sum-exp of A (SURVEY.md section 8a):
//     loss   = (1/2B) sum_ij Pt_ij (rl_i + cl_j - 2 Lg_ij)
//     dLg_ij = (exp(Lg_ij - rl_i) + cs_j exp(Lg_ij - cl_j) - 2 Pt_ij) / 2B,  cs_j = sum_i Pt_ij
//     dA_ij  = Pt_ij (rl_i + cl_j - 2 Lg_ij - wbar_i) / 2B,      wbar_i = sum_j Pt_ij W_ij
//     dS = dLg I / T + (dA + dA^T) S a          dI = dLg^T S / T + (dA + dA^T) I a
// (targets stay in the graph exactly as in the reference: the dA terms are their gradient).
//
// Execution: rows are processed in blocks of R (all of B when it fits the workspace).  When one
// block holds the whole batch, the lean pipeline below runs.  Otherwise (a rank's slice of a
// row-sharded batch, or a batch beyond the scratch budget) each block's tensor-core products give
// the rows P1 = Lg_i., P2 = Lg_.i (= (I_i S^T)/T) and P3 = A_i., with the row log-sum-exp
// partials of each product out of its epilogue; they are merged into rl, cl, za.  A sweep gives
// wbar, cs and the loss, and a third pass the gradient factors, which are written straight into
// TilePack operands and contracted with [I;S]^T / [S;I]^T by two more tensor-core products.  With
// more than one block, phases 2 and 3 recompute each block's products.  All products use the
// 3-term fp16 split (gemm.cu), i.e. fp32-level accuracy: logits reach +-256 here (LayerNorm'd
// embeddings have norm 16), so single-pass fp16/bf16 operands cannot meet the 1e-3 gradient
// tolerance.
#include <algorithm>
#include "common.cuh"
#include "gemm.cuh"
#include "umma.cuh"

namespace mclst {

constexpr int LS_THREADS = 256;

__device__ __forceinline__ float block_sum(float v, float* sh) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = 0.f;
  for (int w = 0; w < LS_THREADS / 32; ++w) r += sh[w];
  __syncthreads();
  return r;
}

// soft targets, sweep 2: wbar_r = sum_j Pt_rj W_rj ; cs_r = sum_j exp(A_rj - za_j)  (A symmetric)
__global__ void __launch_bounds__(LS_THREADS)
soft_pass2_kernel(const float* __restrict__ P1, const float* __restrict__ P3, int64_t ld, int ncols,
                  int64_t row0, const float* __restrict__ rl, const float* __restrict__ cl,
                  const float* __restrict__ za, const float* __restrict__ za_lo,
                  float* __restrict__ wbar, float* __restrict__ cs) {
  __shared__ float sh[LS_THREADS / 32];
  const int64_t r = blockIdx.x, rg = row0 + r;
  const float* p1 = P1 + r * ld;
  const float* p3 = P3 + r * ld;
  const float rl_r = rl[rg], za_r = za[rg], zal_r = za_lo[rg];
  float w = 0.f, c = 0.f;
  auto push = [&](float a, float p1j, int j) {
    w += __expf((a - za_r) - zal_r) * (rl_r + __ldg(cl + j) - 2.f * p1j);
    c += __expf((a - __ldg(za + j)) - __ldg(za_lo + j));
  };
  const int n4 = ((ld & 3) == 0) ? (ncols >> 2) : 0;
  for (int j = threadIdx.x; j < n4; j += LS_THREADS) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(p3) + j);
    const float4 b = __ldg(reinterpret_cast<const float4*>(p1) + j);
    push(a.x, b.x, 4 * j); push(a.y, b.y, 4 * j + 1); push(a.z, b.z, 4 * j + 2); push(a.w, b.w, 4 * j + 3);
  }
  for (int j = n4 * 4 + threadIdx.x; j < ncols; j += LS_THREADS) push(p3[j], p1[j], j);
  w = block_sum(w, sh);
  c = block_sum(c, sh);
  if (threadIdx.x == 0) { wbar[rg] = w; cs[rg] = c; }
}

// loss = (1/2B) sum_r term_r; term = wbar (soft) or rl + cl - 2 diag (eye).  One block.
__global__ void __launch_bounds__(LS_THREADS)
loss_reduce_kernel(const float* __restrict__ a, const float* __restrict__ b,
                   const float* __restrict__ d, const float* __restrict__ a_lo,
                   const float* __restrict__ b_lo, int r_begin, int r_end, int B,
                   float* __restrict__ out) {
  __shared__ double shd[LS_THREADS / 32];
  double acc = 0.0;
  for (int r = r_begin + threadIdx.x; r < r_end; r += LS_THREADS)
    acc += b ? ((double)a[r] + (double)a_lo[r]) + ((double)b[r] + (double)b_lo[r]) - 2.0 * (double)d[r]
             : (double)a[r];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) shd[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < LS_THREADS / 32; ++w) t += shd[w];
    *out = (float)(t / (2.0 * B));
  }
}

struct GradParams {
  const float *P1, *P2, *P3;
  int64_t ld;
  int B, rows, soft;           // rows = valid rows of this block
  int64_t row0;
  const float *rl, *cl, *za, *wbar, *cs, *rl_lo, *cl_lo, *za_lo;
  float inv_t, a_scale;
  uint8_t *ga_hi, *ga_lo, *gb_hi, *gb_lo;   // TilePack A operands, K = [B64 | B64] (soft) or [B64] (eye)
  int nkb_total, nkb_half;
};

__device__ __forceinline__ void store_split(uint8_t* hi, uint8_t* lo, size_t off, const float (&v)[8]) {
  uint32_t h[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const __half a = __float2half_rn(v[2 * i]), b = __float2half_rn(v[2 * i + 1]);
    const __half al = __float2half_rn(v[2 * i] - __half2float(a));
    const __half bl = __float2half_rn(v[2 * i + 1] - __half2float(b));
    h[i] = (uint32_t)__half_as_ushort(a) | ((uint32_t)__half_as_ushort(b) << 16);
    l[i] = (uint32_t)__half_as_ushort(al) | ((uint32_t)__half_as_ushort(bl) << 16);
  }
  *reinterpret_cast<uint4*>(hi + off) = make_uint4(h[0], h[1], h[2], h[3]);
  *reinterpret_cast<uint4*>(lo + off) = make_uint4(l[0], l[1], l[2], l[3]);
}

// Gradient factors of one row block, written as split TilePack operands.  One thread per
// (group of GF_ROWS rows, 8-column chunk): the five per-column statistics of its chunk stay in
// registers while it walks the rows (loading them per element made the kernel LSU-bound: 40 scalar
// loads per 8 elements next to 6 vector loads of data).  Gradients of magnitude ~1/B are scaled
// by 2B before the fp16 split (keeps them in fp16's normal range); the GEMM alpha undoes it.
constexpr int GF_ROWS = 8;
__global__ void __launch_bounds__(256, 2)
grad_factor_kernel(const GradParams p, int64_t rows_pad) {
  const int chunks = p.nkb_half * 8;
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t rgp = t / chunks;
  const int c = (int)(t - rgp * chunks);
  if (rgp * GF_ROWS >= rows_pad) return;
  float rl_j[8], cl_j[8], za_j[8], wb_j[8], cs_j[8], rll_j[8], cll_j[8], zal_j[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int j = c * 8 + i;
    const bool ok = j < p.B;
    rl_j[i] = ok ? __ldg(p.rl + j) : 0.f;
    cl_j[i] = ok ? __ldg(p.cl + j) : 0.f;
    rll_j[i] = ok ? __ldg(p.rl_lo + j) : 0.f;
    cll_j[i] = ok ? __ldg(p.cl_lo + j) : 0.f;
    zal_j[i] = (ok && p.soft) ? __ldg(p.za_lo + j) : 0.f;
    za_j[i] = (ok && p.soft) ? __ldg(p.za + j) : 0.f;
    wb_j[i] = (ok && p.soft) ? __ldg(p.wbar + j) : 0.f;
    cs_j[i] = (ok && p.soft) ? __ldg(p.cs + j) : 1.f;
  }
#pragma unroll 1
  for (int rr = 0; rr < GF_ROWS; ++rr) {
    const int64_t r = rgp * GF_ROWS + rr;
    float g1[8], g2[8], gs[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { g1[i] = 0.f; g2[i] = 0.f; gs[i] = 0.f; }
    if (r < p.rows) {
      const int64_t rg = p.row0 + r;
      const float rl_r = __ldg(p.rl + rg), cl_r = __ldg(p.cl + rg);
      const float rll_r = __ldg(p.rl_lo + rg), cll_r = __ldg(p.cl_lo + rg);
      const float zal_r = p.soft ? __ldg(p.za_lo + rg) : 0.f;
      const float za_r = p.soft ? __ldg(p.za + rg) : 0.f, wb_r = p.soft ? __ldg(p.wbar + rg) : 0.f;
      const float cs_r = p.soft ? __ldg(p.cs + rg) : 1.f;
      // the product rows are B64 wide: two 16-byte loads per array are always in bounds
      float p1v[8], p2v[8], p3v[8];
      const size_t o = (size_t)r * p.ld + (size_t)c * 8;
      *reinterpret_cast<float4*>(p1v) = __ldg(reinterpret_cast<const float4*>(p.P1 + o));
      *reinterpret_cast<float4*>(p1v + 4) = __ldg(reinterpret_cast<const float4*>(p.P1 + o) + 1);
      *reinterpret_cast<float4*>(p2v) = __ldg(reinterpret_cast<const float4*>(p.P2 + o));
      *reinterpret_cast<float4*>(p2v + 4) = __ldg(reinterpret_cast<const float4*>(p.P2 + o) + 1);
      if (p.soft) {
        *reinterpret_cast<float4*>(p3v) = __ldg(reinterpret_cast<const float4*>(p.P3 + o));
        *reinterpret_cast<float4*>(p3v + 4) = __ldg(reinterpret_cast<const float4*>(p.P3 + o) + 1);
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int j = c * 8 + i;
        if (j < p.B) {
          const float p1 = p1v[i], p2 = p2v[i];
          float pt_rj, pt_jr;
          if (p.soft) {
            const float a = p3v[i];
            pt_rj = expf((a - za_r) - zal_r);
            pt_jr = expf((a - za_j[i]) - zal_j[i]);
            const float da_rj = pt_rj * (rl_r + cl_j[i] - 2.f * p1 - wb_r);
            const float da_jr = pt_jr * (rl_j[i] + cl_r - 2.f * p2 - wb_j[i]);
            gs[i] = (da_rj + da_jr) * p.a_scale;
          } else {
            pt_rj = pt_jr = (rg == j) ? 1.f : 0.f;
          }
          g1[i] = (expf((p1 - rl_r) - rll_r) + cs_j[i] * expf((p1 - cl_j[i]) - cll_j[i]) - 2.f * pt_rj) * p.inv_t;   // 2B * dLg_rj / T
          g2[i] = (expf((p2 - rl_j[i]) - rll_j[i]) + cs_r * expf((p2 - cl_r) - cll_r) - 2.f * pt_jr) * p.inv_t;      // 2B * dLg_jr / T
        }
      }
    }
    const size_t off = tilepack_chunk_offset(r, c, p.nkb_total);
    store_split(p.ga_hi, p.ga_lo, off, g1);
    store_split(p.gb_hi, p.gb_lo, off, g2);
    if (p.soft) {
      const size_t off2 = tilepack_chunk_offset(r, p.nkb_half * 8 + c, p.nkb_total);
      store_split(p.ga_hi, p.ga_lo, off2, gs);
      store_split(p.gb_hi, p.gb_lo, off2, gs);
    }
  }
}


// ============================================================================ lean single-block path
// When one row block holds the whole batch, the statistics come out of the product epilogues and
// every element of the products is read ONCE by each consumer:
//   P1 (+ row LSE partials + diagonal from the GEMM epilogue), P3 (+ row LSE partials)
//   column LSE of P1 from a coalesced sweep (replaces the transposed product P2 and its sweep)
//   wbar / cs sweep (soft targets)
//   gradient factors per PAIR of mirrored 64 x 64 tiles: Lg_rj and Lg_jr, A_rj = A_jr are in
//   shared memory together, so each exponential is evaluated once and P3 is read over the upper
//   triangle only; G1 (dLg) and the symmetric Gs are written once each (8 B/element instead of
//   16 + a third product), and dI reads G1 transposed (MN-major tcgen05 descriptors).

// partial (max, sum exp) pairs [slot][ld] -> float-pair statistic per row.  Slot s covers columns
// [s * slot_cols, ...): slots starting at or beyond ncols were never written and are skipped.
// The statistic is kept as a float pair hi + lo (|lo| <= ulp(hi)/2): logits reach +-256 here, where
// one float32 ulp is 3e-5 -- rounding rl / cl / za to a single float puts that much SYSTEMATIC error
// into every exponent of the row and costs the small gradient entries a digit (measured: 1.5e-3
// element-wise vs 1e-4 with the pair).  Consumers form exp((x - hi) - lo).
struct MergeJob { const float2* part; int slots, slot_cols, ncols; int64_t ld; float *hi, *lo; int n; };
struct MergeJobs { MergeJob j[3]; };

__global__ void __launch_bounds__(256)
lse_merge_kernel(const MergeJobs jobs) {
  const MergeJob& J = jobs.j[blockIdx.y];
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= J.n) return;
  // one pass, running maximum in float (exact), sum in double: only the final logarithm and the
  // addition need the extra digits (the pair's lo half is below 2e-5 by construction)
  float M = -INFINITY;
  double S = 0.0;
  for (int s = 0; s < J.slots && (int64_t)s * J.slot_cols < J.ncols; ++s) {
    const float2 p = J.part[(size_t)s * J.ld + r];
    if (p.x > M) { S *= (double)__expf(M - p.x); M = p.x; }
    if (p.x > -INFINITY) S += (double)p.y * (double)__expf(p.x - M);
  }
  const double L = (double)M + log(S);
  const float hi = (float)L;
  J.hi[r] = hi;
  J.lo[r] = (hi == hi && fabsf(hi) < INFINITY) ? (float)(L - (double)hi) : 0.f;
}

// column-wise (max, sum exp) of P [rows, ld] over row chunks of CL_ROWS: thread = column, rows
// streamed with 8 loads in flight; part [chunk][ld].
// rows per chunk: 1024 for large batches, fewer when that would leave the GPU idle (B = 1024: one
// chunk per column block was 4 blocks and 59 us of serial latency)
static int col_chunk_rows(int B) { return B >= 16384 ? 1024 : (B >= 4096 ? 256 : 64); }
__global__ void __launch_bounds__(128)
col_lse_partial_kernel(const float* __restrict__ P, int64_t ld, int rows, int ncols, int chunk_rows,
                       float2* __restrict__ part) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int r0 = blockIdx.y * chunk_rows, r1 = min(rows, r0 + chunk_rows);
  if (j >= ncols) return;
  const float* p = P + j;
  float m = -INFINITY, s = 0.f;
  int r = r0;
  for (; r + 8 <= r1; r += 8) {
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __ldg(p + (size_t)(r + i) * ld);
    float cm = v[0];
#pragma unroll
    for (int i = 1; i < 8; ++i) cm = fmaxf(cm, v[i]);
    if (cm > m) { s *= __expf(m - cm); m = cm; }
#pragma unroll
    for (int i = 0; i < 8; ++i) s += __expf(v[i] - m);
  }
  for (; r < r1; ++r) {
    const float x = __ldg(p + (size_t)r * ld);
    if (x > m) { s = s * __expf(m - x) + 1.f; m = x; }
    else s += __expf(x - m);
  }
  part[(size_t)blockIdx.y * ld + j] = make_float2(m, s);
}

struct TileGradParams {
  const float *P1, *P3;
  int64_t ld;
  int B, soft;
  const float *rl, *cl, *za, *wbar, *cs, *rl_lo, *cl_lo, *za_lo;
  float inv_t, a_scale;            // normalised so that the stored factors are O(1)
  uint8_t *g1_hi, *g1_lo, *gs_hi, *gs_lo;   // TilePack images [rows_pad, B64], K = batch index
  int nkb;                         // B64 / 64
};

// (exponentials here and in the sweeps use the ex2.approx path: 2 ulp, and the argument's own
// rounding |a| 2^-24 only matters where exp(a) is negligible)
constexpr int TG = 64;             // tile edge
constexpr int TG_LD = TG + 1;
constexpr int TG_SMEM = (3 * TG * TG_LD + 2 * 8 * TG) * 4;

__global__ void __launch_bounds__(256, 4)
grad_tiles_kernel(const TileGradParams p) {
  const int tr = blockIdx.y, tc = blockIdx.x;
  if (tc < tr) return;                                   // the pair (tr, tc) also serves (tc, tr)
  extern __shared__ float tg_smem[];
  float* sA = tg_smem;                                   // P1[tr rows][tc cols]
  float* sB = sA + TG * TG_LD;                           // P1[tc rows][tr cols]   -> later g_jr
  float* sC = sB + TG * TG_LD;                           // P3[tr rows][tc cols]   -> later h
  float* st_r = sC + TG * TG_LD;                         // [8][64] statistics of the tr indices
  float* st_c = st_r + 8 * TG;                           // [8][64] statistics of the tc indices
  const int t = threadIdx.x;
  const int64_t R0 = (int64_t)tr * TG, C0 = (int64_t)tc * TG;
  // ---- load the three tiles (coalesced float4 rows) and the 2 x 64 x 8 statistics
  for (int q = t; q < TG * TG / 4; q += 256) {
    const int r = q >> 4, c4 = (q & 15) * 4;
    const float4 a = __ldg(reinterpret_cast<const float4*>(p.P1 + (R0 + r) * p.ld + C0 + c4));
    sA[r * TG_LD + c4] = a.x; sA[r * TG_LD + c4 + 1] = a.y; sA[r * TG_LD + c4 + 2] = a.z; sA[r * TG_LD + c4 + 3] = a.w;
    const float4 b = __ldg(reinterpret_cast<const float4*>(p.P1 + (C0 + r) * p.ld + R0 + c4));
    sB[r * TG_LD + c4] = b.x; sB[r * TG_LD + c4 + 1] = b.y; sB[r * TG_LD + c4 + 2] = b.z; sB[r * TG_LD + c4 + 3] = b.w;
    if (p.soft) {
      const float4 c = __ldg(reinterpret_cast<const float4*>(p.P3 + (R0 + r) * p.ld + C0 + c4));
      sC[r * TG_LD + c4] = c.x; sC[r * TG_LD + c4 + 1] = c.y; sC[r * TG_LD + c4 + 2] = c.z; sC[r * TG_LD + c4 + 3] = c.w;
    }
  }
  if (t < 2 * TG) {
    const int i = t & (TG - 1);
    const int64_t g = ((t < TG) ? R0 : C0) + i;
    float* d = (t < TG) ? st_r : st_c;
    const bool ok = g < p.B;
    d[0 * TG + i] = ok ? __ldg(p.rl + g) : 0.f;
    d[1 * TG + i] = ok ? __ldg(p.cl + g) : 0.f;
    d[2 * TG + i] = ok ? __ldg(p.rl_lo + g) : 0.f;
    d[3 * TG + i] = ok ? __ldg(p.cl_lo + g) : 0.f;
    d[4 * TG + i] = (ok && p.soft) ? __ldg(p.za + g) : 0.f;
    d[5 * TG + i] = (ok && p.soft) ? __ldg(p.za_lo + g) : 0.f;
    d[6 * TG + i] = (ok && p.soft) ? __ldg(p.wbar + g) : 0.f;
    d[7 * TG + i] = (ok && p.soft) ? __ldg(p.cs + g) : 1.f;
  }
  __syncthreads();
  // ---- thread (r, 16-column quarter): the 16 (r, j) pairs; both orientations from one set of exps
  const int r = t >> 2, jq = (t & 3) * 16;
  const int64_t R = R0 + r;
  const float rl_r = st_r[r], cl_r = st_r[TG + r], rll_r = st_r[2 * TG + r], cll_r = st_r[3 * TG + r];
  const float za_r = st_r[4 * TG + r], zal_r = st_r[5 * TG + r], wb_r = st_r[6 * TG + r], cs_r = st_r[7 * TG + r];
  float g_rj[16], g_jr[16], h[16];
#pragma unroll
  for (int u = 0; u < 16; ++u) {
    const int j = jq + u;
    const int64_t J = C0 + j;
    float a1 = 0.f, a2 = 0.f, hh = 0.f;
    if (R < p.B && J < p.B) {
      const float x = sA[r * TG_LD + j], y = sB[j * TG_LD + r];
      const float rl_j = st_c[j], cl_j = st_c[TG + j], rll_j = st_c[2 * TG + j], cll_j = st_c[3 * TG + j];
      float p_rj, p_jr;
      if (p.soft) {
        const float a = sC[r * TG_LD + j];
        p_rj = __expf((a - za_r) - zal_r);
        p_jr = __expf((a - st_c[4 * TG + j]) - st_c[5 * TG + j]);
        const float da_rj = p_rj * (rl_r + cl_j - 2.f * x - wb_r);
        const float da_jr = p_jr * (rl_j + cl_r - 2.f * y - st_c[6 * TG + j]);
        hh = (da_rj + da_jr) * p.a_scale;
      } else {
        p_rj = p_jr = (R == J) ? 1.f : 0.f;
      }
      a1 = (__expf((x - rl_r) - rll_r) + st_c[7 * TG + j] * __expf((x - cl_j) - cll_j) - 2.f * p_rj) * p.inv_t;   // 2B dLg_rj / T
      a2 = (__expf((y - rl_j) - rll_j) + cs_r * __expf((y - cl_r) - cll_r) - 2.f * p_jr) * p.inv_t;               // 2B dLg_jr / T
    }
    g_rj[u] = a1; g_jr[u] = a2; h[u] = hh;
  }
  // as-is tile (tr, tc): row R, K chunks (C0 + jq) / 8 and the next one
  {
    const int chunk0 = (int)((C0 + jq) >> 3);
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      const size_t off = tilepack_chunk_offset(R, chunk0 + half, p.nkb);
      float v[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = g_rj[half * 8 + i];
      store_split(p.g1_hi, p.g1_lo, off, v);
      if (p.soft) {
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = h[half * 8 + i];
        store_split(p.gs_hi, p.gs_lo, off, v);
      }
    }
  }
  if (tc == tr) return;                                  // (block-uniform)
  // ---- mirrored tile (tc, tr): transpose the two result tiles through shared memory
  __syncthreads();                                       // everyone has read sA / sB / sC
#pragma unroll
  for (int u = 0; u < 16; ++u) {
    sB[r * TG_LD + jq + u] = g_jr[u];
    sC[r * TG_LD + jq + u] = h[u];
  }
  __syncthreads();
  {
    const int j = t >> 2, rq = (t & 3) * 16;             // row C0 + j of the mirrored tile, columns R0 + rq ..
    const int64_t J = C0 + j;
    const int chunk0 = (int)((R0 + rq) >> 3);
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      const size_t off = tilepack_chunk_offset(J, chunk0 + half, p.nkb);
      float v[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = sB[(rq + half * 8 + i) * TG_LD + j];      // dLg_jr as row j
      store_split(p.g1_hi, p.g1_lo, off, v);
      if (p.soft) {
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = sC[(rq + half * 8 + i) * TG_LD + j];
        store_split(p.gs_hi, p.gs_lo, off, v);
      }
    }
  }
}

// ---------------------------------------------------------------------------- host plan
struct LossPlan {
  int B, D, soft;
  int64_t B64, R, nblocks;
  uint32_t* flags;
  PackedOperand Sp, Ip, ISp;       // rows padded to 256: usable as A and as B operands
  PackedOperand XT_IS, XT_SI;      // [D, 2*B64] (soft) or [D, B64] (eye), transposed packs
  PackedOperand GA, GB;            // [R, 2*B64] / [R, B64]
  float *P1, *P2, *P3;
  float *rl, *cl, *za, *wbar, *cs, *diag, *rl_lo, *cl_lo, *za_lo;   // views into the stats block [9][B]
  float* stats_ws;
  size_t bytes;
  bool lean;                       // one row block holds the whole batch
  PackedOperand G1, Gs;            // lean: [R, B64] each
  // LSE partials: rows of P1 / P2 / P3 [2 * nt256][R] (P2 general, partc lean), columns of P1 [chunks][B64]
  float2 *part1, *part2, *part3, *partc;
  int nt256, cchunks;
};

static LossPlan plan_loss(void* ws, size_t cap, int B, int D, int soft, size_t budget, int64_t rows_local) {
  LossPlan L{};
  L.B = B; L.D = D; L.soft = soft;
  L.B64 = (int64_t)align_up((size_t)B, 64);
  // row-block size: P1,P2,P3 (12 B/elem) + GA,GB hi/lo (8 or 16 B/elem) per (row, column)
  const size_t per_row = (size_t)L.B64 * (12 + (soft ? 16 : 8));
  int64_t R = (int64_t)(budget / std::max<size_t>(per_row, 1));
  R = std::max<int64_t>(128, R / 128 * 128);
  R = std::min<int64_t>(R, (int64_t)align_up((size_t)rows_local, 128));
  L.R = R;
  L.nblocks = ceil_div(rows_local, R);
  L.lean = L.nblocks == 1 && rows_local == B;
  L.nt256 = (int)ceil_div(B, 256);
  L.cchunks = (int)ceil_div(B, col_chunk_rows(B));
  Arena a(ws, cap);
  L.flags = a.take<uint32_t>(16);
  L.Sp = take_operand(a, B, D, true, true, 1);
  L.Ip = take_operand(a, B, D, true, true, 1);
  if (soft) L.ISp = take_operand(a, B, 2 * (int64_t)align_up((size_t)D, 64), true, true, 1);
  const int64_t kx = (soft ? 2 : 1) * L.B64;
  L.XT_IS = take_operand(a, D, kx, true, true, 1);
  L.XT_SI = take_operand(a, D, kx, true, true, 1);
  if (L.lean) {
    L.G1 = take_operand(a, R, L.B64, false, true, 1);
    if (soft) L.Gs = take_operand(a, R, L.B64, false, true, 1);
  } else {
    L.GA = take_operand(a, R, kx, false, true, 1);
    L.GB = take_operand(a, R, kx, false, true, 1);
  }
  L.P1 = a.take<float>((size_t)R * L.B64);
  L.P2 = L.lean ? nullptr : a.take<float>((size_t)R * L.B64);
  L.P3 = soft ? a.take<float>((size_t)R * L.B64) : nullptr;
  L.part1 = a.take<float2>((size_t)2 * L.nt256 * R);
  L.part3 = soft ? a.take<float2>((size_t)2 * L.nt256 * R) : nullptr;
  if (L.lean) L.partc = a.take<float2>((size_t)L.cchunks * L.B64);
  else L.part2 = a.take<float2>((size_t)2 * L.nt256 * R);
  L.stats_ws = a.take<float>((size_t)MCLST_LOSS_STAT_ROWS * B);
  L.bytes = align_up(a.off, 256);
  return L;
}

// Row-block scratch budget.  A B200 has 180 GB: by default up to 32 GiB may be spent so that
// batches up to 32k rows need a single row block (no recomputation of the three products per
// sweep); smaller budgets stream the batch in row blocks.
static size_t loss_budget() {
  const char* e = getenv("MCLST_LOSS_SCRATCH_MB");
  return (size_t)(e ? atoll(e) : 32768) << 20;
}

// rows [i0, i0+rows) of P1 = S I^T / T, P2 = I S^T / T (need_p2), P3 = [I|S][I|S]^T * a, each with
// its row log-sum-exp partials (part1 / part2 / part3, rows indexed locally) and P1 with its diagonal
// out of the product epilogue.  The fused statistics fix the tile shape (gemm_variant), so a block
// that phases 2 and 3 recompute is bit-identical to the one phase 1 took rl, cl, za from: the
// softmax weights exp(A - za) of the recomputed rows then sum to one as exactly as in phase 1.
static int compute_blocks(const LossPlan& L, int64_t i0, int64_t rows, float inv_t, float a_scale,
                          bool need_p2, cudaStream_t st) {
  const int nkbD = L.Sp.nkb;
  GemmParams g{};
  g.nseg = 3; g.batch = 1; g.M = rows; g.N = L.B; g.ldc = L.B64;
  g.amax_bits = L.flags; g.amax_pow = 2;          // both operands carry the tensor-wide factor
  const size_t a_off = (size_t)(i0 / 128) * nkbD * TP_SLICE_BYTES;
  int rc;
  g.nkb = nkbD;
  g.a_hi = L.Sp.hi + a_off; g.a_lo = L.Sp.lo + a_off; g.b_hi = L.Ip.hi; g.b_lo = L.Ip.lo;
  g.c = L.P1; g.alpha = inv_t;
  g.lse_part = L.part1; g.lse_ld = L.R; g.diag = L.diag + i0; g.diag_offset = i0;
  if ((rc = launch_gemm_tn(g, st))) return rc;
  g.diag = nullptr;
  if (need_p2) {
    g.a_hi = L.Ip.hi + a_off; g.a_lo = L.Ip.lo + a_off; g.b_hi = L.Sp.hi; g.b_lo = L.Sp.lo;
    g.c = L.P2; g.lse_part = L.part2;
    if ((rc = launch_gemm_tn(g, st))) return rc;
  }
  if (L.soft) {
    const size_t a2 = (size_t)(i0 / 128) * L.ISp.nkb * TP_SLICE_BYTES;
    g.nkb = L.ISp.nkb;
    g.a_hi = L.ISp.hi + a2; g.a_lo = L.ISp.lo + a2; g.b_hi = L.ISp.hi; g.b_lo = L.ISp.lo;
    g.c = L.P3; g.alpha = a_scale; g.lse_part = L.part3;
    if ((rc = launch_gemm_tn(g, st))) return rc;
  }
  return 0;
}

static void bind_stats(LossPlan& L, float* stats) {
  const size_t B = (size_t)L.B;
  L.rl = stats; L.cl = stats + B; L.za = stats + 2 * B; L.wbar = stats + 3 * B; L.cs = stats + 4 * B;
  L.diag = stats + 5 * B;
  L.rl_lo = stats + 6 * B; L.cl_lo = stats + 7 * B; L.za_lo = stats + 8 * B;
}

// One phase of the loss for the rows [row0, row0 + rows) of the (all-gathered) batch.
//   phase 1: pack operands; rl, cl, za (+ diag) of the local rows
//   phase 2: wbar, cs of the local rows (soft targets; needs every rank's rl, cl, za)
//   phase 3: local loss contribution and the gradients of the local rows (needs all stats)
static int loss_phase(const float* spot_emb, int64_t ld_s, const float* image_emb, int64_t ld_i,
                      int B, int D, float temperature, int target_mode, int64_t row0, int64_t rows,
                      int phase, float* stats, float* loss_out, float* d_spot, int64_t ld_ds,
                      float* d_image, int64_t ld_di, void* workspace, size_t workspace_bytes,
                      cudaStream_t st) {
  const int soft = target_mode != MCLST_T_EYE;
  const float inv_t = 1.0f / temperature;
  const float a_scale = target_mode == MCLST_T_SOFT_DIV ? 0.5f / temperature
                      : target_mode == MCLST_T_SOFT_MUL ? 0.5f * temperature : 0.f;
  LossPlan L = plan_loss(workspace, workspace_bytes, B, D, soft, loss_budget(), rows);
  MCLST_REQUIRE(L.bytes <= workspace_bytes, MCLST_ERR_WORKSPACE, "contrastive_loss: workspace %zu < %zu",
                workspace_bytes, L.bytes);
  bind_stats(L, stats ? stats : L.stats_ws);
  int rc;
  const int nkbD = L.Sp.nkb;
  // one row block holds every row this call owns (the whole batch, or this rank's slice of it):
  // P1 / P2 / P3 survive in the workspace between the phases and nothing is recomputed
  const bool single = L.nblocks == 1;
  if (phase == 1) {
    // one power-of-two factor for both embedding matrices (they are concatenated along K and
    // shared between products): max|x| over S and I as a device word every consumer reads
    MCLST_CUDA(cudaMemsetAsync(L.flags, 0, 64, st));
    prof_mark(st, "loss_pack");
    if ((rc = launch_amax_bits(spot_emb, B, D, ld_s, L.flags, st))) return rc;
    if ((rc = launch_amax_bits(image_emb, B, D, ld_i, L.flags, st))) return rc;
    if ((rc = launch_pack_split(spot_emb, B, D, ld_s, false, 1.f, L.Sp, 0, nkbD, L.flags, nullptr, st))) return rc;
    if ((rc = launch_pack_split(image_emb, B, D, ld_i, false, 1.f, L.Ip, 0, nkbD, L.flags, nullptr, st))) return rc;
    if (soft) {
      if ((rc = launch_pack_split(image_emb, B, D, ld_i, false, 1.f, L.ISp, 0, nkbD, L.flags, nullptr, st))) return rc;
      if ((rc = launch_pack_split(spot_emb, B, D, ld_s, false, 1.f, L.ISp, nkbD, nkbD, L.flags, nullptr, st))) return rc;
    }
    if (d_spot) {
      const int nkbB = (int)(L.B64 / 64);
      if ((rc = launch_pack_split(image_emb, B, D, ld_i, true, 1.f, L.XT_IS, 0, nkbB, L.flags, nullptr, st))) return rc;
      if ((rc = launch_pack_split(spot_emb, B, D, ld_s, true, 1.f, L.XT_SI, 0, nkbB, L.flags, nullptr, st))) return rc;
      if (soft) {
        if ((rc = launch_pack_split(spot_emb, B, D, ld_s, true, 1.f, L.XT_IS, nkbB, nkbB, L.flags, nullptr, st))) return rc;
        if ((rc = launch_pack_split(image_emb, B, D, ld_i, true, 1.f, L.XT_SI, nkbB, nkbB, L.flags, nullptr, st))) return rc;
      }
    }
    // products with the row statistics fused into their epilogues, then one merge per row block.
    // Lean: no transposed product; the column statistics come from a sweep over P1 instead.
    for (int64_t b = 0; b < L.nblocks; ++b) {
      const int64_t i0 = row0 + b * L.R, nr = std::min<int64_t>(L.R, row0 + rows - i0);
      if ((rc = compute_blocks(L, i0, nr, inv_t, a_scale, !L.lean, st))) return rc;
      MergeJobs mj{};
      mj.j[0] = MergeJob{L.part1, 2 * L.nt256, 128, B, L.R, L.rl + i0, L.rl_lo + i0, (int)nr};
      if (L.lean) {
        prof_mark(st, "col_lse");
        col_lse_partial_kernel<<<dim3((unsigned)ceil_div(B, 128), (unsigned)L.cchunks), 128, 0, st>>>(
            L.P1, L.B64, B, B, col_chunk_rows(B), L.partc);
        MCLST_LAUNCH_CHECK();
        mj.j[1] = MergeJob{L.partc, L.cchunks, 1, L.cchunks, L.B64, L.cl, L.cl_lo, B};
      } else {
        mj.j[1] = MergeJob{L.part2, 2 * L.nt256, 128, B, L.R, L.cl + i0, L.cl_lo + i0, (int)nr};
      }
      if (soft) mj.j[2] = MergeJob{L.part3, 2 * L.nt256, 128, B, L.R, L.za + i0, L.za_lo + i0, (int)nr};
      prof_mark(st, "lse_merge");
      lse_merge_kernel<<<dim3((unsigned)ceil_div(nr, 256), soft ? 3u : 2u), 256, 0, st>>>(mj);
      MCLST_LAUNCH_CHECK();
    }
  } else if (phase == 2) {
    if (soft) {
      for (int64_t b = 0; b < L.nblocks; ++b) {
        const int64_t i0 = row0 + b * L.R, nr = std::min<int64_t>(L.R, row0 + rows - i0);
        if (!single && (rc = compute_blocks(L, i0, nr, inv_t, a_scale, false, st))) return rc;
        prof_mark(st, "soft_pass2");
        soft_pass2_kernel<<<(unsigned)nr, LS_THREADS, 0, st>>>(L.P1, L.P3, L.B64, B, i0, L.rl, L.cl,
                                                             L.za, L.za_lo, L.wbar, L.cs);
        MCLST_LAUNCH_CHECK();
      }
    }
  } else {
    prof_mark(st, "loss_reduce");
    if (soft) loss_reduce_kernel<<<1, LS_THREADS, 0, st>>>(L.wbar, nullptr, nullptr, nullptr, nullptr, (int)row0, (int)(row0 + rows), B, loss_out);
    else loss_reduce_kernel<<<1, LS_THREADS, 0, st>>>(L.rl, L.cl, L.diag, L.rl_lo, L.cl_lo, (int)row0, (int)(row0 + rows), B, loss_out);
    MCLST_LAUNCH_CHECK();
    if (d_spot && L.lean) {
      const float u = std::max(inv_t, a_scale);
      TileGradParams tp{};
      tp.P1 = L.P1; tp.P3 = L.P3; tp.ld = L.B64; tp.B = B; tp.soft = soft;
      tp.rl = L.rl; tp.cl = L.cl; tp.za = L.za; tp.wbar = L.wbar; tp.cs = L.cs;
      tp.rl_lo = L.rl_lo; tp.cl_lo = L.cl_lo; tp.za_lo = L.za_lo;
      tp.inv_t = inv_t / u; tp.a_scale = a_scale / u;
      tp.g1_hi = L.G1.hi; tp.g1_lo = L.G1.lo;
      tp.gs_hi = L.Gs.hi; tp.gs_lo = L.Gs.lo; tp.nkb = L.G1.nkb;
      static bool attr_set = false;
      if (!attr_set) {
        MCLST_CUDA(cudaFuncSetAttribute(grad_tiles_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TG_SMEM));
        attr_set = true;
      }
      const unsigned nt = (unsigned)ceil_div(B, TG);
      prof_mark(st, "grad_tiles");
      grad_tiles_kernel<<<dim3(nt, nt), 256, TG_SMEM, st>>>(tp);
      MCLST_LAUNCH_CHECK();
      GemmParams g{};
      g.nseg = 3; g.batch = 1; g.M = B; g.N = D; g.alpha = 0.5f * u / (float)B;
      g.amax_bits = L.flags; g.amax_pow = 1;
      g.nkb = (soft ? 2 : 1) * L.G1.nkb;
      if (soft) { g.a_nkb1 = L.G1.nkb; g.a2_hi = L.Gs.hi; g.a2_lo = L.Gs.lo; }
      g.a_hi = L.G1.hi; g.a_lo = L.G1.lo; g.b_hi = L.XT_IS.hi; g.b_lo = L.XT_IS.lo;
      g.c = d_spot; g.ldc = ld_ds;
      // dS and dI are independent and, for small batches, a few tiles each (B = 1024: 8 CTAs walking
      // K = 2048 for 47 us): side by side on two streams
      const bool pair = ceil_div(B, 128) * ceil_div(D, 256) * 2 <= sm_count();
      cudaStream_t s2 = st;
      if (pair && (rc = side_fork(st, &s2))) return rc;
      if ((rc = launch_gemm_tn(g, st))) return rc;
      // dI = dLg^T S + Gs I reads the dLg image TRANSPOSED (MN-major tcgen05 descriptors) instead of
      // a second, transposed copy of it (4 more bytes per element for the factor kernel to write)
      g.a1_mn = L.G1.nkb;
      g.a_nkb1 = L.G1.nkb;                   // (eye targets: image 1 is the whole K range)
      g.b_hi = L.XT_SI.hi; g.b_lo = L.XT_SI.lo;
      g.c = d_image; g.ldc = ld_di;
      if ((rc = launch_gemm_tn(g, s2))) return rc;
      if (pair) prof_mark(s2, "end");
      if (pair && (rc = side_join(st))) return rc;
    } else if (d_spot) {
      for (int64_t b = 0; b < L.nblocks; ++b) {
        const int64_t i0 = row0 + b * L.R, nr = std::min<int64_t>(L.R, row0 + rows - i0);
        if (!single && (rc = compute_blocks(L, i0, nr, inv_t, a_scale, true, st))) return rc;
        GradParams gp{};
        gp.P1 = L.P1; gp.P2 = L.P2; gp.P3 = L.P3; gp.ld = L.B64; gp.B = B; gp.rows = (int)nr;
        gp.soft = soft; gp.row0 = i0; gp.rl = L.rl; gp.cl = L.cl; gp.za = L.za; gp.wbar = L.wbar;
        // the two K halves carry different scalars (1/T and a); the larger one goes into alpha so that
        // the stored factors stay O(1) whatever the temperature (fp16 range)
        const float u = std::max(inv_t, a_scale);
        gp.rl_lo = L.rl_lo; gp.cl_lo = L.cl_lo; gp.za_lo = L.za_lo;
        gp.cs = L.cs; gp.inv_t = inv_t / u; gp.a_scale = a_scale / u;
        gp.ga_hi = L.GA.hi; gp.ga_lo = L.GA.lo; gp.gb_hi = L.GB.hi; gp.gb_lo = L.GB.lo;
        gp.nkb_total = L.GA.nkb; gp.nkb_half = (int)(L.B64 / 64);
        const int64_t rows_pad = (int64_t)align_up((size_t)nr, 128);
        const int64_t threads = rows_pad / GF_ROWS * gp.nkb_half * 8;
        prof_mark(st, "grad_factor");
        grad_factor_kernel<<<(unsigned)ceil_div(threads, 256), 256, 0, st>>>(gp, rows_pad);
        MCLST_LAUNCH_CHECK();
        GemmParams g{};
        g.nseg = 3; g.batch = 1; g.M = nr; g.N = D; g.nkb = L.GA.nkb; g.alpha = 0.5f * u / (float)B;
        g.amax_bits = L.flags; g.amax_pow = 1;    // only the embedding operand is scaled
        g.a_hi = L.GA.hi; g.a_lo = L.GA.lo; g.b_hi = L.XT_IS.hi; g.b_lo = L.XT_IS.lo;
        g.c = d_spot + (i0 - row0) * ld_ds; g.ldc = ld_ds;
        if ((rc = launch_gemm_tn(g, st))) return rc;
        g.a_hi = L.GB.hi; g.a_lo = L.GB.lo; g.b_hi = L.XT_SI.hi; g.b_lo = L.XT_SI.lo;
        g.c = d_image + (i0 - row0) * ld_di; g.ldc = ld_di;
        if ((rc = launch_gemm_tn(g, st))) return rc;
      }
    }
    prof_mark(st, "end");
  }
  return 0;
}

}  // namespace mclst

using namespace mclst;

extern "C" int mclst_contrastive_loss_workspace_bytes(int batch, int dim, int target_mode,
                                                      int64_t rows_local, size_t* bytes) {
  MCLST_REQUIRE(bytes && batch >= 1 && dim >= 1 && target_mode >= 0 && target_mode <= 2 &&
                rows_local >= 1 && rows_local <= batch, MCLST_ERR_INVALID,
                "contrastive_loss_workspace: bad args");
  *bytes = plan_loss(nullptr, 0, batch, dim, target_mode != MCLST_T_EYE, loss_budget(), rows_local).bytes;
  return 0;
}

static int check_loss_args(const float* s, const float* i, int batch, int dim, float t, int mode,
                           const void* ws) {
  MCLST_REQUIRE(s && i && ws, MCLST_ERR_INVALID, "contrastive_loss: null pointer");
  MCLST_REQUIRE(batch >= 1 && dim >= 1 && t > 0.f, MCLST_ERR_INVALID,
                "contrastive_loss: bad batch/dim/temperature");
  MCLST_REQUIRE(mode >= 0 && mode <= 2, MCLST_ERR_INVALID, "contrastive_loss: bad target mode");
  return 0;
}

extern "C" int mclst_contrastive_loss(const float* spot_emb, int64_t ld_s, const float* image_emb,
                                      int64_t ld_i, int batch, int dim, float temperature,
                                      int target_mode, float* loss_out, float* d_spot,
                                      int64_t ld_ds, float* d_image, int64_t ld_di,
                                      void* workspace, size_t workspace_bytes,
                                      mclst_stream_t stream) {
  int rc;
  if ((rc = check_loss_args(spot_emb, image_emb, batch, dim, temperature, target_mode, workspace))) return rc;
  MCLST_REQUIRE(loss_out, MCLST_ERR_INVALID, "contrastive_loss: null loss_out");
  MCLST_REQUIRE((d_spot == nullptr) == (d_image == nullptr), MCLST_ERR_INVALID,
                "contrastive_loss: pass both gradients or neither");
  cudaStream_t st = (cudaStream_t)stream;
  for (int phase = 1; phase <= 3; ++phase)
    if ((rc = loss_phase(spot_emb, ld_s, image_emb, ld_i, batch, dim, temperature, target_mode, 0, batch,
                         phase, nullptr, loss_out, d_spot, ld_ds, d_image, ld_di, workspace,
                         workspace_bytes, st))) return rc;
  return 0;
}

extern "C" int mclst_contrastive_loss_phase(const float* spot_emb, int64_t ld_s,
                                            const float* image_emb, int64_t ld_i, int batch, int dim,
                                            float temperature, int target_mode, int64_t row0,
                                            int64_t rows, int phase, float* stats, float* loss_out,
                                            float* d_spot, int64_t ld_ds, float* d_image,
                                            int64_t ld_di, void* workspace, size_t workspace_bytes,
                                            mclst_stream_t stream) {
  int rc;
  if ((rc = check_loss_args(spot_emb, image_emb, batch, dim, temperature, target_mode, workspace))) return rc;
  MCLST_REQUIRE(stats && phase >= 1 && phase <= 3, MCLST_ERR_INVALID, "contrastive_loss_phase: bad phase/stats");
  MCLST_REQUIRE(row0 >= 0 && rows >= 1 && row0 + rows <= batch && row0 % 128 == 0, MCLST_ERR_INVALID,
                "contrastive_loss_phase: row range [%lld, +%lld) must start on a multiple of 128",
                (long long)row0, (long long)rows);
  MCLST_REQUIRE(phase != 3 || loss_out, MCLST_ERR_INVALID, "contrastive_loss_phase: null loss_out");
  return loss_phase(spot_emb, ld_s, image_emb, ld_i, batch, dim, temperature, target_mode, row0, rows,
                    phase, stats, loss_out, d_spot, ld_ds, d_image, ld_di, workspace, workspace_bytes,
                    (cudaStream_t)stream);
}
