// Split-precision tcgen05 GEMM:  C[M,N] = epilogue(alpha * A[M,K] * B[N,K]^T)
//
// The reference computes every contraction of the path in FP32 (cuBLAS sgemm with TF32
// off, SURVEY.md 2a).  Tensor cores take 16-bit operands, so each fp32 operand x is split
// at pack time into two fp16 TilePack images hi = fp16(x), lo = fp16(x - hi) and the
// product is accumulated over three K segments
//       A_hi*B_hi + A_lo*B_hi + A_hi*B_lo        (the lo*lo term is < 2^-22 relative)
// in the fp32 TMEM accumulator: ~fp32 accuracy at 3 tensor-core passes.  nseg = 1 gives a
// plain fp16 product.
//
//   pack_split      fp32 row-major -> (hi, lo) TilePack, optionally transposed, written at a
//                   K offset so operands can be concatenated along K
//   gemm_tn         one CTA per 128 x 256 output tile: warp 0 streams A/B slices with
//                   cp.async.bulk into a 4-stage ring, warp 1 issues tcgen05.mma, warps 2-5
//                   run the epilogue out of TMEM (alpha, bias, exact-erf GELU, residual).
//
// Operand scale: fp16 has a 5-bit exponent (overflow at 65504, subnormal below 6.1e-5), so every
// operand is brought to the top of that range with an EXACT power-of-two factor before the split
// and the factor is undone in the epilogue:
//   * generic matmul: one factor per operand row (its largest |x| lands in [1, 2)), found by the
//     pack kernel itself; the epilogue multiplies element (m, n) by inv_a[m] * inv_b[n];
//   * operands that are concatenated along K or shared between products (the loss): one factor for
//     the whole tensor, derived by every consumer from a device-side max|x| word (amax_bits).
// Anything smaller than 2^-25 of its row's largest entry is lost, i.e. the error stays relative to
// the row scale at fp32 level whatever the magnitude of the data (1e-30 .. 1e+30).  Non-finite
// inputs are not scaled and propagate as inf/NaN exactly as in an fp32 product.
#include <algorithm>
#include <cstdlib>
#include "common.cuh"
#include "gemm.cuh"
#include "umma.cuh"

namespace mclst {

using namespace ptx;

// ============================================================================ pack_split
// power-of-two factor 2^(1-e) that maps amax = m * 2^e (m in [0.5, 1)) into [1, 2); 1 for zero or
// non-finite amax.  *inv receives the exact inverse.
__device__ __forceinline__ float pow2_scale(float amax, float* inv) {
  if (!(amax > 0.f) || !(amax < INFINITY)) { *inv = 1.f; return 1.f; }
  int e;
  frexpf(amax, &e);
  e = max(-125, min(126, e));
  *inv = ldexpf(1.f, e - 1);
  return ldexpf(1.f, 1 - e);
}
__device__ __forceinline__ void split8(const float (&v)[8], uint4* h, uint4* l) {
  uint32_t hh[4], ll[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const __half a = __float2half_rn(v[2 * i]), b = __float2half_rn(v[2 * i + 1]);
    const __half al = __float2half_rn(v[2 * i] - __half2float(a));
    const __half bl = __float2half_rn(v[2 * i + 1] - __half2float(b));
    hh[i] = (uint32_t)__half_as_ushort(a) | ((uint32_t)__half_as_ushort(b) << 16);
    ll[i] = (uint32_t)__half_as_ushort(al) | ((uint32_t)__half_as_ushort(bl) << 16);
  }
  *h = make_uint4(hh[0], hh[1], hh[2], hh[3]);
  *l = make_uint4(ll[0], ll[1], ll[2], ll[3]);
}

// Non-transposed: out row r = in row r, K index = in column.  One warp per row.
// inv_scale != null: per-row factor (computed here, inverse stored); else amax_bits != null: the
// tensor-wide factor; else none.
__device__ __forceinline__ void
pack_plain_block(const float* __restrict__ x, int64_t rows, int64_t cols, int64_t ld,
                 float scale, uint8_t* __restrict__ hi, uint8_t* __restrict__ lo,
                 int64_t rows_pad, int nkb_total, int kb_offset, int nkb_mine,
                 const uint32_t* __restrict__ amax_bits, float* __restrict__ inv_scale,
                 int64_t x_batch, size_t out_batch, unsigned bx, unsigned bz) {
  x += (int64_t)bz * x_batch;
  hi += (size_t)bz * out_batch;
  if (lo) lo += (size_t)bz * out_batch;
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)bx * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= rows_pad) return;
  float inv = 1.f;
  if (inv_scale && nkb_mine <= 16 && kb_offset == 0) {
    // the whole row in registers (K <= 1024): ONE round trip to memory instead of eight dependent
    // ones (max scan, then chunk by chunk) -- the pack of a training-step operand is pure latency
    float v[4][8];
    float amax = 0.f;
    // 16-byte loads when the rows allow it: a lane's chunk is 32 contiguous bytes, and eight scalar
    // loads per chunk made the pack (pure latency at these sizes) issue four times the instructions
    const bool vec = (ld % 4 == 0) && (((uintptr_t)x & 15) == 0) && (x_batch % 4 == 0);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = lane + 32 * j;
      const int64_t k0 = (int64_t)c * 8;
      if (vec && r < rows && k0 + 8 <= cols) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(x + r * ld + k0));
        const float4 b = __ldg(reinterpret_cast<const float4*>(x + r * ld + k0) + 1);
        v[j][0] = a.x; v[j][1] = a.y; v[j][2] = a.z; v[j][3] = a.w;
        v[j][4] = b.x; v[j][5] = b.y; v[j][6] = b.z; v[j][7] = b.w;
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int64_t k = k0 + i;
          v[j][i] = (r < rows && k < cols) ? __ldg(x + r * ld + k) : 0.f;
        }
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int i = 0; i < 8; ++i) amax = fmaxf(amax, fabsf(v[j][i]));
    amax = warp_max(amax);
    scale *= pow2_scale(amax, &inv);
    if (lane == 0) inv_scale[(size_t)bz * rows_pad + r] = inv;
    const int nchunks = nkb_mine * 8;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = lane + 32 * j;
      if (c < nchunks) {
        float w[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) w[i] = v[j][i] * scale;
        uint4 h, l;
        split8(w, &h, &l);
        const size_t off = tilepack_chunk_offset(r, c, nkb_total);
        *reinterpret_cast<uint4*>(hi + off) = h;
        if (lo) *reinterpret_cast<uint4*>(lo + off) = l;
      }
    }
    return;
  }
  if (inv_scale) {
    float amax = 0.f;
    if (r < rows) {
      const float* row = x + r * ld;
      int64_t k = lane;
      for (; k + 7 * 32 < cols; k += 8 * 32) {          // 8 independent loads in flight
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = __ldg(row + k + 32 * i);
#pragma unroll
        for (int i = 0; i < 8; ++i) amax = fmaxf(amax, fabsf(v[i]));
      }
      for (; k < cols; k += 32) amax = fmaxf(amax, fabsf(__ldg(row + k)));
    }
    amax = warp_max(amax);
    scale *= pow2_scale(amax, &inv);
    if (lane == 0) inv_scale[(size_t)bz * rows_pad + r] = inv;
  } else if (amax_bits) {
    scale *= pow2_scale(__uint_as_float(__ldg(amax_bits)), &inv);
  }
  const int nchunks = nkb_mine * 8;
  for (int c = lane; c < nchunks; c += 32) {
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int64_t k = (int64_t)c * 8 + i;
      v[i] = (r < rows && k < cols) ? __ldg(x + r * ld + k) * scale : 0.f;
    }
    uint4 h, l;
    split8(v, &h, &l);
    const size_t off = tilepack_chunk_offset(r, kb_offset * 8 + c, nkb_total);
    *reinterpret_cast<uint4*>(hi + off) = h;
    if (lo) *reinterpret_cast<uint4*>(lo + off) = l;
  }
}

__global__ void __launch_bounds__(256)
pack_split_kernel(const float* __restrict__ x, int64_t rows, int64_t cols, int64_t ld,
                  float scale, uint8_t* __restrict__ hi, uint8_t* __restrict__ lo,
                  int64_t rows_pad, int nkb_total, int kb_offset, int nkb_mine,
                  const uint32_t* __restrict__ amax_bits, float* __restrict__ inv_scale,
                  int64_t x_batch, size_t out_batch) {
  pack_plain_block(x, rows, cols, ld, scale, hi, lo, rows_pad, nkb_total, kb_offset, nkb_mine, amax_bits,
                   inv_scale, x_batch, out_batch, blockIdx.x, blockIdx.z);
}

// Transposed: out row r = in column r, K index = in row.  Lane <-> out row (contiguous in
// the input), each thread gathers 8 consecutive K (8 input rows) for one 16-byte chunk.
// With inv_scale the block first scans its 32 columns for their max|x| (gridDim.y must be 1; the
// block then has 32 warps and keeps 8 independent loads in flight per thread: a serial scan of a
// 1024-row column cost 70 us per pack and 1.2 ms per training step).
__device__ __forceinline__ void
pack_trans_block(const float* __restrict__ x, int64_t rows, int64_t cols, int64_t ld,
                 float scale, uint8_t* __restrict__ hi, uint8_t* __restrict__ lo,
                 int64_t out_rows_pad, int nkb_total, int kb_offset, int nkb_mine,
                 const uint32_t* __restrict__ amax_bits, float* __restrict__ inv_scale,
                 int64_t x_batch, size_t out_batch, unsigned bx, unsigned by, unsigned ny, unsigned bz,
                 float (*s_amax)[32]) {
  x += (int64_t)bz * x_batch;
  hi += (size_t)bz * out_batch;
  if (lo) lo += (size_t)bz * out_batch;
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)bx * 32 + lane;                            // out row = in column
  const int cgroup = threadIdx.x >> 5;                                  // chunk lane
  const int ngroups = blockDim.x >> 5;                                  // 8 (y-split grid) or 32 (self-scaling)
  float inv = 1.f;
  if (inv_scale && nkb_mine <= 16 && kb_offset == 0 && ngroups == 32 && ny == 1) {
    // the thread's four chunks (32 input rows of its column) in registers: one round trip
    float v[4][8];
    float amax = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = cgroup + 32 * j;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int64_t k = (int64_t)c * 8 + i;
        v[j][i] = (r < cols && k < rows) ? __ldg(x + k * ld + r) : 0.f;
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int i = 0; i < 8; ++i) amax = fmaxf(amax, fabsf(v[j][i]));
    s_amax[cgroup][lane] = amax;
    __syncthreads();
    for (int g = 0; g < 32; ++g) amax = fmaxf(amax, s_amax[g][lane]);
    scale *= pow2_scale(amax, &inv);
    if (cgroup == 0 && r < out_rows_pad) inv_scale[(size_t)bz * out_rows_pad + r] = inv;
    if (r >= out_rows_pad) return;
    const int nchunks = nkb_mine * 8;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = cgroup + 32 * j;
      if (c < nchunks) {
        float w[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) w[i] = v[j][i] * scale;
        uint4 h, l;
        split8(w, &h, &l);
        const size_t off = tilepack_chunk_offset(r, c, nkb_total);
        *reinterpret_cast<uint4*>(hi + off) = h;
        if (lo) *reinterpret_cast<uint4*>(lo + off) = l;
      }
    }
    return;
  }
  if (inv_scale) {
    float amax = 0.f;
    if (r < cols) {
      const float* col = x + r;
      int64_t k = cgroup;
      for (; k + 7 * ngroups < rows; k += 8 * ngroups) {
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = __ldg(col + (k + i * ngroups) * ld);
#pragma unroll
        for (int i = 0; i < 8; ++i) amax = fmaxf(amax, fabsf(v[i]));
      }
      for (; k < rows; k += ngroups) amax = fmaxf(amax, fabsf(__ldg(col + k * ld)));
    }
    s_amax[cgroup][lane] = amax;
    __syncthreads();
    for (int g = 0; g < ngroups; ++g) amax = fmaxf(amax, s_amax[g][lane]);
    scale *= pow2_scale(amax, &inv);
    if (cgroup == 0 && r < out_rows_pad) inv_scale[(size_t)bz * out_rows_pad + r] = inv;
  } else if (amax_bits) {
    scale *= pow2_scale(__uint_as_float(__ldg(amax_bits)), &inv);
  }
  if (r >= out_rows_pad) return;
  const int nchunks = nkb_mine * 8;
  for (int c = by * ngroups + cgroup; c < nchunks; c += ny * ngroups) {
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int64_t k = (int64_t)c * 8 + i;                             // in row
      v[i] = (r < cols && k < rows) ? __ldg(x + k * ld + r) * scale : 0.f;
    }
    uint4 h, l;
    split8(v, &h, &l);
    const size_t off = tilepack_chunk_offset(r, kb_offset * 8 + c, nkb_total);
    *reinterpret_cast<uint4*>(hi + off) = h;
    if (lo) *reinterpret_cast<uint4*>(lo + off) = l;
  }
}

__global__ void __launch_bounds__(1024)
pack_split_t_kernel(const float* __restrict__ x, int64_t rows, int64_t cols, int64_t ld,
                    float scale, uint8_t* __restrict__ hi, uint8_t* __restrict__ lo,
                    int64_t out_rows_pad, int nkb_total, int kb_offset, int nkb_mine,
                    const uint32_t* __restrict__ amax_bits, float* __restrict__ inv_scale,
                    int64_t x_batch, size_t out_batch) {
  __shared__ float s_amax[32][32];
  pack_trans_block(x, rows, cols, ld, scale, hi, lo, out_rows_pad, nkb_total, kb_offset, nkb_mine, amax_bits,
                   inv_scale, x_batch, out_batch, blockIdx.x, blockIdx.y, gridDim.y, blockIdx.z, s_amax);
}

// Both operands of one matmul in ONE launch (the training step is launch-bound: 51 products, two
// packs each): blocks [0, a.blocks) pack A, the rest pack B, each plain or transposed, 32 warps,
// per-row factors.
struct PackJob {
  const float* x;
  int64_t rows, cols, ld, rows_pad, x_batch;
  uint8_t *hi, *lo;
  float* inv_scale;
  size_t out_batch;
  int nkb, transpose, blocks_x, blocks;      // blocks = blocks_x * batch
};
__global__ void __launch_bounds__(1024)
pack_pair_kernel(const PackJob a, const PackJob b) {
  __shared__ float s_amax[32][32];
  const bool first = blockIdx.x < (unsigned)a.blocks;
  const PackJob& j = first ? a : b;
  const unsigned id = first ? blockIdx.x : blockIdx.x - (unsigned)a.blocks;
  const unsigned bx = id % (unsigned)j.blocks_x, bz = id / (unsigned)j.blocks_x;
  if (j.transpose)
    pack_trans_block(j.x, j.rows, j.cols, j.ld, 1.f, j.hi, j.lo, j.rows_pad, j.nkb, 0, j.nkb, nullptr,
                     j.inv_scale, j.x_batch, j.out_batch, bx, 0, 1, bz, s_amax);
  else
    pack_plain_block(j.x, j.rows, j.cols, j.ld, 1.f, j.hi, j.lo, j.rows_pad, j.nkb, 0, j.nkb, nullptr,
                     j.inv_scale, j.x_batch, j.out_batch, bx, bz);
}

static PackJob make_pack_job(const float* x, int64_t rows, int64_t cols, int64_t ld, bool transpose,
                             const PackedOperand& dst, int batch, int64_t x_batch_elems, int rows_per_block = 32) {
  PackJob j{};
  j.x = x; j.rows = rows; j.cols = cols; j.ld = ld; j.rows_pad = dst.rows_pad; j.x_batch = x_batch_elems;
  j.hi = dst.hi; j.lo = dst.lo; j.inv_scale = dst.inv_scale; j.out_batch = dst.bytes; j.nkb = dst.nkb;
  j.transpose = transpose ? 1 : 0;
  j.blocks_x = (int)ceil_div(dst.rows_pad, rows_per_block);   // plain: one row per warp; transposed: 32 columns per block
  j.blocks = j.blocks_x * batch;
  return j;
}

int launch_pack_pair(const float* A, int64_t a_rows, int64_t a_cols, int64_t lda, bool a_trans,
                     const PackedOperand& pa, int64_t a_batch_elems, const float* B, int64_t b_rows,
                     int64_t b_cols, int64_t ldb, bool b_trans, const PackedOperand& pb,
                     int64_t b_batch_elems, int batch, cudaStream_t st) {
  // two plain operands (every forward Linear): 8 rows per block instead of 32 -- 64 blocks of 1024
  // threads left more than half of the SMs idle in a kernel that is one load-compute-store latency
  // chain; the transposed pack needs its 32 warps (column maxima across 32 K groups)
  const int threads = (!a_trans && !b_trans) ? 256 : 1024;
  const PackJob ja = make_pack_job(A, a_rows, a_cols, lda, a_trans, pa, batch, a_batch_elems, threads / 32);
  const PackJob jb = make_pack_job(B, b_rows, b_cols, ldb, b_trans, pb, batch, b_batch_elems, threads / 32);
  pack_pair_kernel<<<(unsigned)(ja.blocks + jb.blocks), threads, 0, st>>>(ja, jb);
  MCLST_LAUNCH_CHECK();
  return 0;
}

// max|x| of a tensor as the bit pattern of a non-negative float (orders like an unsigned integer);
// *out must be zeroed by the caller.  NaNs are ignored (fmaxf), +-inf is kept.
__global__ void __launch_bounds__(256)
amax_bits_kernel(const float* __restrict__ x, int64_t rows, int64_t cols, int64_t ld,
                 uint32_t* __restrict__ out) {
  float amax = 0.f;
  const int64_t total = rows * cols;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / cols, c = i - r * cols;
    amax = fmaxf(amax, fabsf(__ldg(x + r * ld + c)));
  }
  amax = warp_max(amax);
  if ((threadIdx.x & 31) == 0 && amax > 0.f) atomicMax(out, __float_as_uint(amax));
}

int launch_amax_bits(const float* x, int64_t rows, int64_t cols, int64_t ld, uint32_t* out, cudaStream_t st) {
  const int64_t total = rows * cols;
  const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(ceil_div(total, 256 * 8), (int64_t)sm_count() * 8));
  amax_bits_kernel<<<grid, 256, 0, st>>>(x, rows, cols, ld, out);
  MCLST_LAUNCH_CHECK();
  return 0;
}

int launch_pack_split(const float* x, int64_t rows, int64_t cols, int64_t ld, bool transpose,
                      float scale, const PackedOperand& dst, int kb_offset, int nkb_mine,
                      const uint32_t* amax_bits, float* inv_scale, cudaStream_t st, int batch,
                      int64_t x_batch_elems) {
  if (!transpose) {
    const int wpb = 8;
    dim3 grid((unsigned)ceil_div(dst.rows_pad, wpb), 1, (unsigned)batch);
    pack_split_kernel<<<grid, wpb * 32, 0, st>>>(x, rows, cols, ld, scale, dst.hi, dst.lo,
                                                 dst.rows_pad, dst.nkb, kb_offset, nkb_mine, amax_bits,
                                                 inv_scale, x_batch_elems, dst.bytes);
  } else {
    dim3 grid((unsigned)ceil_div(dst.rows_pad, 32), inv_scale ? 1u : (unsigned)std::min<int64_t>(64, nkb_mine),
              (unsigned)batch);
    pack_split_t_kernel<<<grid, inv_scale ? 1024 : 256, 0, st>>>(x, rows, cols, ld, scale, dst.hi, dst.lo,
                                              dst.rows_pad, dst.nkb, kb_offset, nkb_mine, amax_bits,
                                              inv_scale, x_batch_elems, dst.bytes);
  }
  MCLST_LAUNCH_CHECK();
  return 0;
}

// ============================================================================ gemm_tn
#ifdef GM_TIMING
__device__ unsigned long long g_gm_dbg[16];
#define GM_STAMP(slot) do { if (blockIdx.x == 0) g_gm_dbg[slot] = ptx::globaltimer(); } while (0)
#else
#define GM_STAMP(slot) do {} while (0)
#endif
constexpr int GM_EPI_WARPS = 8;                              // two per TMEM lane quadrant, 4 column chunks each
constexpr int GM_THREADS = 64 + 32 * GM_EPI_WARPS;
constexpr int GM_BM = 128, GM_BN = 256;
constexpr int GM_STAGES = 4;
constexpr int GM_STAGE_BYTES = 3 * TP_SLICE_BYTES;     // A slice (128 rows) + B slice (256 rows)
constexpr int GM_EPI_BYTES = GM_EPI_WARPS * 32 * 32 * 4;                // one 32x32 fp32 transpose tile per epilogue warp
constexpr int GM_SMEM = GM_STAGES * GM_STAGE_BYTES + 1024 + GM_EPI_BYTES + 1024;

__device__ __forceinline__ float gelu_erf(float x) {
  return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
}

// Persistent: every CTA walks output tiles with the same three roles as sim_topk (TMA producer /
// single-thread MMA issuer / 8 epilogue warps) and a double-buffered 2 x 256-column TMEM
// accumulator, so the epilogue of tile i (TMEM -> registers -> 128 KiB of global stores) overlaps
// the MMAs of tile i+1.
// CL = 2: the two CTAs of a cluster take vertically adjacent 128-row tiles of the same 256-column
// strip; each fetches half of every B slice and multicasts it to both.  With both operands
// streamed a 128x256 tile needs 87 FLOP per byte from L2 (16 TB/s at full tensor rate, more than
// L2 delivers: the CL = 1 kernel measured ~500 TFLOP/s on the loss products); sharing B cuts the
// traffic per CTA from 48 to 32 KiB per K block.
// BN = 128 halves the tile: a problem with fewer than one 128 x 256 tile per SM (every nn.Linear of
// the B = 1024 training step: 32 .. 48 tiles on 148 SMs) is bounded by the serial K loop of ONE
// tile, and a 128-column tile walks it in half the time while twice as many SMs take part.
template <int CL, int BN>
__global__ void __launch_bounds__(GM_THREADS, 1)
gemm_tn_kernel(const GemmParams p) {
  static_assert(BN == 256 || ((BN == 128 || BN == 64) && CL == 1), "tile widths: 256, or 128 / 64 without B sharing");
  constexpr int STAGE_TX = (1 + BN / 128) * TP_SLICE_BYTES;
  // The half-width kernel serves the small problems, and those are L2-bound, not tensor-bound: 96
  // CTAs re-streaming 32 KiB per 256 MMA cycles ask L2 for > 20 TB/s (CUPTI timeline of the graphed
  // training step: 26 us per product where the MMAs need 7).  It therefore loads the hi AND lo slice
  // of both operands ONCE per K block (64 KiB stage, 3 stages) and issues all three split products
  // from them, instead of streaming a 32 KiB stage per (segment, K block): a third less L2 traffic.
  // BN = 64 (quarter width) once even 128-wide tiles leave half of the SMs idle: per tile the K loop
  // is bound by the per-SM L2 -> shared-memory rate (116 GB/s: 8.9 us for 16 K blocks of 64 KiB) and
  // the drain by the per-SM store rate (3.0 us for 64 KiB), so twice as many SMs with 48 / 32 KiB
  // each finish sooner (globaltimer stamps, tools/gemm_timing.py).  The B half tile is the first or
  // second 8 KiB of a TilePack slice (8 of its 16 swizzle atoms).
  constexpr bool FUSE = BN <= 128;
  constexpr int B_BYTES = (BN == 64) ? TP_SLICE_BYTES / 2 : TP_SLICE_BYTES;
  constexpr int NSTAGE = FUSE ? 3 : GM_STAGES;
  constexpr int STAGE_BYTES = FUSE ? 4 * TP_SLICE_BYTES : GM_STAGE_BYTES;
  static_assert(NSTAGE * STAGE_BYTES == GM_STAGES * GM_STAGE_BYTES, "same shared-memory footprint");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* bar_full = reinterpret_cast<uint64_t*>(smem + GM_STAGES * GM_STAGE_BYTES);
  uint64_t* bar_empty = bar_full + GM_STAGES;
  uint64_t* bar_tfull = bar_empty + GM_STAGES;
  uint64_t* bar_tempty = bar_tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_tempty + 2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkb = p.nkb;
  const int iters = p.nseg * nkb;
  const int mt = (int)((p.M + GM_BM - 1) / GM_BM), nt = (int)((p.N + BN - 1) / BN);
  const int mg = (mt + CL - 1) / CL;                     // groups of CL vertically adjacent tiles
  const int64_t groups = (int64_t)mg * nt * p.batch;
  const uint32_t crank = (CL > 1) ? cluster_ctarank() : 0u;
  const int64_t g0 = blockIdx.x / CL, gstep = gridDim.x / CL;
  constexpr uint16_t kMask = (uint16_t)((1u << CL) - 1u);

  if (threadIdx.x == 0) GM_STAMP(0);
  if (threadIdx.x == 0) {
    for (int i = 0; i < GM_STAGES; ++i) { mbar_init(&bar_full[i], 1); mbar_init(&bar_empty[i], CL); }
    for (int i = 0; i < 2; ++i) { mbar_init(&bar_tfull[i], 1); mbar_init(&bar_tempty[i], GM_EPI_WARPS); }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  if (CL > 1) cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) GM_STAMP(1);

  if (warp == 0) {
    if (lane == 0) {
      const uint64_t pol = policy_evict_last();
      uint32_t stage = 0, phase = 0;
      for (int64_t g = g0; g < groups; g += gstep) {
        const int mb = min((int)(g % mg) * CL + (int)crank, mt - 1);     // ghost tiles re-read the last block
        const int nb = (int)((g / mg) % nt), z = (int)(g / ((int64_t)mg * nt));
        const uint8_t* a_hi = p.a_hi + (size_t)z * p.a_batch_bytes;
        const uint8_t* a_lo = p.a_lo ? p.a_lo + (size_t)z * p.a_batch_bytes : nullptr;
        const uint8_t* b_hi = p.b_hi + (size_t)z * p.b_batch_bytes;
        const uint8_t* b_lo = p.b_lo ? p.b_lo + (size_t)z * p.b_batch_bytes : nullptr;
        if (FUSE) {
          for (int kb = 0; kb < nkb; ++kb) {
            mbar_wait(&bar_empty[stage], phase ^ 1);
            mbar_arrive_expect_tx(&bar_full[stage], (p.nseg == 3 ? 2 : 1) * (TP_SLICE_BYTES + B_BYTES));
            uint8_t* dst = smem + stage * STAGE_BYTES;
            const size_t ao = ((size_t)mb * nkb + kb) * TP_SLICE_BYTES;
            const size_t bo = (BN == 64) ? ((size_t)(nb >> 1) * nkb + kb) * TP_SLICE_BYTES + (size_t)(nb & 1) * B_BYTES
                                         : ((size_t)nb * nkb + kb) * TP_SLICE_BYTES;
            bulk_g2s(dst, a_hi + ao, TP_SLICE_BYTES, &bar_full[stage]);
            bulk_g2s(dst + 2 * TP_SLICE_BYTES, b_hi + bo, B_BYTES, &bar_full[stage]);
            if (p.nseg == 3) {
              bulk_g2s(dst + TP_SLICE_BYTES, a_lo + ao, TP_SLICE_BYTES, &bar_full[stage]);
              bulk_g2s(dst + 3 * TP_SLICE_BYTES, b_lo + bo, B_BYTES, &bar_full[stage]);
            }
            if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
          }
          continue;
        }
        for (int it = 0; it < iters; ++it) {
          const int seg = it / nkb, kb = it - seg * nkb;
          // segment 0: hi*hi, 1: lo*hi, 2: hi*lo
          const uint8_t* a = (seg == 1) ? a_lo : a_hi;
          const uint8_t* b = (seg == 2) ? b_lo : b_hi;
          // A may be two images concatenated along K (the second one shared between products)
          size_t a_off = ((size_t)mb * nkb + kb) * TP_SLICE_BYTES;
          if (p.a_nkb1 > 0) {
            if (kb < p.a_nkb1) a_off = ((size_t)mb * p.a_nkb1 + kb) * TP_SLICE_BYTES;
            else {
              a = (seg == 1) ? p.a2_lo : p.a2_hi;
              a_off = ((size_t)mb * (nkb - p.a_nkb1) + (kb - p.a_nkb1)) * TP_SLICE_BYTES;
            }
          }
          mbar_wait(&bar_empty[stage], phase ^ 1);
          mbar_arrive_expect_tx(&bar_full[stage], STAGE_TX);
          uint8_t* dst = smem + stage * GM_STAGE_BYTES;
          if (p.a1_mn > 0 && kb < p.a_nkb1) {
            // transposed image: 64 of its rows (K') x the 128 columns of output tile mb = the lower
            // or upper 8 atoms of two neighbouring K slices of row block kb / 2
            const uint8_t* img = (seg == 1) ? a_lo : a_hi;
            const int s0 = 2 * mb, s1 = min(2 * mb + 1, p.a1_mn - 1);
            const size_t rb_off = (size_t)(kb >> 1) * p.a1_mn;
            const size_t half = (size_t)(kb & 1) * (TP_SLICE_BYTES / 2);
            bulk_g2s(dst, img + (rb_off + s0) * TP_SLICE_BYTES + half, TP_SLICE_BYTES / 2, &bar_full[stage]);
            bulk_g2s(dst + TP_SLICE_BYTES / 2, img + (rb_off + s1) * TP_SLICE_BYTES + half, TP_SLICE_BYTES / 2,
                     &bar_full[stage]);
          } else
          bulk_g2s(dst, a + a_off, TP_SLICE_BYTES, &bar_full[stage]);
          if (BN == 128) {
            bulk_g2s(dst + TP_SLICE_BYTES, b + ((size_t)nb * nkb + kb) * TP_SLICE_BYTES,
                     TP_SLICE_BYTES, &bar_full[stage]);
          } else if (CL == 1) {
            bulk_g2s(dst + TP_SLICE_BYTES, b + ((size_t)(2 * nb) * nkb + kb) * TP_SLICE_BYTES,
                     TP_SLICE_BYTES, &bar_full[stage]);
            bulk_g2s(dst + 2 * TP_SLICE_BYTES, b + ((size_t)(2 * nb + 1) * nkb + kb) * TP_SLICE_BYTES,
                     TP_SLICE_BYTES, &bar_full[stage]);
          } else {
            // this CTA fetches row block 2 nb + crank of B and multicasts it to the pair
            bulk_g2s_mcast(dst + (1 + crank) * TP_SLICE_BYTES,
                           b + ((size_t)(2 * nb + crank) * nkb + kb) * TP_SLICE_BYTES, TP_SLICE_BYTES,
                           &bar_full[stage], kMask, pol);
          }
          if (++stage == GM_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // uniform control flow for the whole warp, one elected lane issues (umma.cuh: elect_one)
    constexpr uint32_t idesc = make_idesc_f16(GM_BM, BN, false);
    const uint32_t leader = elect_one();
    uint32_t stage = 0, phase = 0;
    int n = 0;
    for (int64_t g = g0; g < groups; g += gstep, ++n) {
      const int buf = n & 1;
      mbar_wait(&bar_tempty[buf], ((n >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + buf * BN;
      if (FUSE) {
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&bar_full[stage], phase);
          if (lane == 0 && kb == 0) GM_STAMP(2);
          tc_fence_after();
          const uint32_t base = smem_u32(smem + stage * STAGE_BYTES);
          if (leader) {
            for (int seg = 0; seg < p.nseg; ++seg) {          // hi*hi, lo*hi, hi*lo from the same slices
              const uint32_t a_addr = base + (seg == 1 ? TP_SLICE_BYTES : 0);
              const uint32_t b_addr = base + 2 * TP_SLICE_BYTES + (seg == 2 ? TP_SLICE_BYTES : 0);
#pragma unroll
              for (int k4 = 0; k4 < 4; ++k4)
                mma_f16_ss(d_tmem, make_smem_desc_sw128(a_addr + k4 * 32), make_smem_desc_sw128(b_addr + k4 * 32),
                           idesc, (kb | seg | k4) != 0 ? 1u : 0u);
            }
            mma_commit(&bar_empty[stage]);
          }
          __syncwarp();
          if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
        }
        if (leader) mma_commit(&bar_tfull[buf]);
        __syncwarp();
        if (lane == 0) GM_STAMP(3);
        continue;
      }
      for (int it = 0; it < iters; ++it) {
        mbar_wait(&bar_full[stage], phase);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(smem + stage * GM_STAGE_BYTES);
        const uint32_t b_addr = a_addr + TP_SLICE_BYTES;
        const int kb_it = it % nkb;
        if (leader) {
          if (p.a1_mn > 0 && kb_it < p.a_nkb1) {
            // A read MN-major: 16 K' = two 8-row atoms (2 KiB) per instruction; the two 64-column
            // halves of the tile lie 8 KiB apart
#pragma unroll
            for (int k4 = 0; k4 < 4; ++k4)
              mma_f16_ss(d_tmem, make_smem_desc_sw128_mn(a_addr + k4 * 2048, TP_SLICE_BYTES / 2, 1024),
                         make_smem_desc_sw128(b_addr + k4 * 32), idesc_a_mn_major(idesc), (it | k4) != 0 ? 1u : 0u);
          } else {
#pragma unroll
            for (int k4 = 0; k4 < 4; ++k4)
              mma_f16_ss(d_tmem, make_smem_desc_sw128(a_addr + k4 * 32),
                         make_smem_desc_sw128(b_addr + k4 * 32), idesc, (it | k4) != 0 ? 1u : 0u);
          }
          if (CL == 1) mma_commit(&bar_empty[stage]);
          else mma_commit_mcast(&bar_empty[stage], kMask);
        }
        __syncwarp();
        if (++stage == GM_STAGES) { stage = 0; phase ^= 1; }
      }
      if (leader) mma_commit(&bar_tfull[buf]);
      __syncwarp();
    }
  } else {
    // ------------------------------------------------------------ epilogue
    // tcgen05.ld hands every thread one ROW of the chunk; storing that directly makes each warp
    // store touch 32 different 128-byte lines (measured: 1.3 TB/s on the 4 GiB loss products).
    // Each warp therefore transposes its 32x32 chunk through an XOR-swizzled shared tile and
    // stores 4 full 128-byte row segments per instruction.
    const int quad = warp & 3;
    const int chalf = (warp - 2) >> 2;                     // which half of the 8 column chunks
    float4* tile = reinterpret_cast<float4*>(smem + GM_STAGES * GM_STAGE_BYTES + 1024) + (warp - 2) * 256;
    const bool vec_ok = (p.ldc % 4 == 0) && ((uintptr_t)p.c % 16 == 0) && (p.c_batch_elems % 4 == 0) &&
                        (!p.residual || (uintptr_t)p.residual % 16 == 0);
    const int sub = lane >> 3, c4 = lane & 7;              // store phase: row it*4+sub, columns c4*4..+3
    float alpha = p.alpha;
    if (p.amax_bits) {                                     // undo the tensor-wide operand factor(s)
      float inv;
      pow2_scale(__uint_as_float(__ldg(p.amax_bits)), &inv);
      alpha *= (p.amax_pow == 2) ? inv * inv : inv;
    }
    int n = 0;
    for (int64_t g = g0; g < groups; g += gstep, ++n) {
      const int mb = (int)(g % mg) * CL + (int)crank;
      const int nb = (int)((g / mg) % nt), z = (int)(g / ((int64_t)mg * nt));
      const int buf = n & 1;
      const int64_t m0 = (int64_t)mb * GM_BM + quad * 32;
      float* cbase = p.c + (size_t)z * p.c_batch_elems;
      const float* rbase = p.residual ? p.residual + (size_t)z * p.c_batch_elems : nullptr;
      float rs[8];                                         // alpha * per-row operand factor of my 8 store rows
#pragma unroll
      for (int it = 0; it < 8; ++it)
        rs[it] = alpha * ((p.a_scale && mb < mt) ? __ldg(p.a_scale + (size_t)z * p.a_scale_batch + m0 + it * 4 + sub) : 1.f);
      // bias and per-column operand factors of this warp's chunks: fetched BEFORE the accumulator
      // is waited for (inside the chunk loop each of them was an exposed L2 round trip: the epilogue
      // of a 128 x 128 tile took 3.0 us of a 13.8 us kernel -- globaltimer stamps, tools/gemm_timing.py)
      constexpr int NC = BN / 64;
      const int64_t n0 = (int64_t)nb * BN;
      float pbias[NC][4], pcs[NC][4];
#pragma unroll
      for (int u = 0; u < NC; ++u) {
        const int64_t col = n0 + (chalf * NC + u) * 32 + c4 * 4;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          pbias[u][i] = (p.bias && col + i < p.N) ? __ldg(p.bias + col + i) : 0.f;
          // (b_scale is padded to the tile width: always in bounds)
          pcs[u][i] = p.b_scale ? __ldg(p.b_scale + (size_t)z * p.b_scale_batch + col + i) : 1.f;
        }
      }
      mbar_wait(&bar_tfull[buf], (n >> 1) & 1);
      if (threadIdx.x == 64) GM_STAMP(4);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + buf * BN;
      // fused row log-sum-exp (loss products): running (max, sum exp) of MY row (TMEM lane) over
      // the 128 columns this warp drains, written as one partial per (row, tile column, half)
      float lm = -INFINITY, ls = 0.f;
      const int64_t my_row = m0 + lane;
#pragma unroll 1
      for (int c = chalf * (BN / 64); c < (chalf + 1) * (BN / 64); ++c) {
        if (n0 + c * 32 >= p.N || mb >= mt || m0 >= p.M) break;             // uniform
        uint32_t v[32];
        tmem_ld_32x32(taddr + c * 32, v);
        tmem_ld_wait();
        if (threadIdx.x == 64 && c == chalf * (BN / 64)) GM_STAMP(8);
        if (p.lse_part) {
          // 6 instructions per element: scale + max, then subtract + scale + ex2 + add.  The running
          // maximum is taken on the scaled values themselves (exact), so the exponent arguments are
          // small differences; ex2.approx adds 2 ulp to terms that only matter near the maximum.
          const int64_t cbase = n0 + c * 32;
          const bool full = cbase + 32 <= p.N;
          float x[32];
          float cm = -INFINITY;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            x[j] = __uint_as_float(v[j]) * alpha;
            if (!full && cbase + j >= p.N) x[j] = -INFINITY;
            cm = fmaxf(cm, x[j]);
          }
          if (p.diag) {                                   // the one chunk of this warp that crosses the diagonal
            const int64_t dj = my_row + p.diag_offset - cbase;
            if (__any_sync(0xffffffffu, dj >= 0 && dj < 32)) {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (dj == j && my_row < p.M) p.diag[my_row] = x[j];
            }
          }
          if (cm > lm) { ls *= exp2f((lm - cm) * 1.4426950408889634f); lm = cm; }   // (0 on the first chunk)
          if (lm > -INFINITY) {
            float acc0 = 0.f, acc1 = 0.f;
#pragma unroll
            for (int j = 0; j < 32; j += 2) {
              acc0 += exp2f((x[j] - lm) * 1.4426950408889634f);
              acc1 += exp2f((x[j + 1] - lm) * 1.4426950408889634f);
            }
            ls += acc0 + acc1;
          }
          if (!p.c) continue;                                                // statistics only: nothing to store
        }
#pragma unroll
        for (int j = 0; j < 8; ++j)
          tile[lane * 8 + (j ^ (lane & 7))] =
              make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                          __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
        __syncwarp();
        if (threadIdx.x == 64 && c == chalf * (BN / 64)) GM_STAMP(9);
        const int64_t col = n0 + c * 32 + c4 * 4;
        const bool full4 = vec_ok && col + 4 <= p.N;
        float bias[4], cs[4];
        const int cc = c - chalf * NC;                     // (selects with compile-time indices: registers)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float bv = pbias[0][i], cv = pcs[0][i];
          if (NC > 1 && cc == 1) { bv = pbias[1 % NC][i]; cv = pcs[1 % NC][i]; }
          if (NC > 2 && cc == 2) { bv = pbias[2 % NC][i]; cv = pcs[2 % NC][i]; }
          if (NC > 3 && cc == 3) { bv = pbias[3 % NC][i]; cv = pcs[3 % NC][i]; }
          bias[i] = bv;
          cs[i] = cv;
        }
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const int row = it * 4 + sub;
          const float4 t = tile[row * 8 + (c4 ^ (row & 7))];
          const int64_t m = m0 + row;
          if (m >= p.M) continue;
          const float ra = rs[it];
          float o[4] = {t.x * (ra * cs[0]) + bias[0], t.y * (ra * cs[1]) + bias[1],
                        t.z * (ra * cs[2]) + bias[2], t.w * (ra * cs[3]) + bias[3]};
          if (p.act == 1) {
#pragma unroll
            for (int i = 0; i < 4; ++i) o[i] = gelu_erf(o[i]);
          }
          float* crow = cbase + m * p.ldc + col;
          if (full4) {
            float4 w = make_float4(o[0], o[1], o[2], o[3]);
            if (rbase) {
              const float4 rr = *reinterpret_cast<const float4*>(rbase + m * p.ldc + col);
              w.x += rr.x; w.y += rr.y; w.z += rr.z; w.w += rr.w;
            }
            *reinterpret_cast<float4*>(crow) = w;
          } else {
#pragma unroll
            for (int i = 0; i < 4; ++i)
              if (col + i < p.N) crow[i] = o[i] + (rbase ? rbase[m * p.ldc + col + i] : 0.f);
          }
        }
        if (threadIdx.x == 64 && c == chalf * (BN / 64)) GM_STAMP(10);
        __syncwarp();
      }
      if (p.lse_part && mb < mt && my_row < p.M && n0 + chalf * 128 < p.N)
        p.lse_part[(size_t)(nb * 2 + chalf) * p.lse_ld + my_row] = make_float2(lm, ls);
      // accumulator drained: hand the buffer back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (threadIdx.x == 64) GM_STAMP(5);
      if (lane == 0) mbar_arrive(&bar_tempty[buf]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) GM_STAMP(6);
  if (CL > 1) cluster_sync_all();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
  if (threadIdx.x == 32) GM_STAMP(7);
}

template <int CL, int BN>
static int launch_gemm_cl(const GemmParams& q, cudaStream_t st) {
  auto kern = gemm_tn_kernel<CL, BN>;
  static bool attr_set = false;
  if (!attr_set) {
    MCLST_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, GM_SMEM));
    attr_set = true;
  }
  const int64_t mt = ceil_div(q.M, GM_BM), nt = ceil_div(q.N, BN);
  const int64_t groups = ceil_div(mt, CL) * nt * q.batch;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(CL * std::min<int64_t>(groups, sm_count() / CL)));
  cfg.blockDim = dim3(GM_THREADS);
  cfg.dynamicSmemBytes = GM_SMEM;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CL;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  MCLST_CUDA(cudaLaunchKernelEx(&cfg, kern, q));
  MCLST_LAUNCH_CHECK();
  return 0;
}

// Which gemm_tn instantiation a product with an M x N x batch output runs on: *cluster = 2 (CTA pairs
// sharing B, 128 x 256 tiles) or 1, *width = the tile width 256, 128 or 64.  narrow_ok is false for
// products that need 256-wide tiles (fused row statistics, A concatenated along K).
// MCLST_GEMM_CLUSTER=2 forces pairs, any other non-zero value forbids them.
void gemm_variant(int64_t M, int64_t N, int batch, bool narrow_ok, int* cluster, int* width) {
  static const int force = [] { const char* e = getenv("MCLST_GEMM_CLUSTER"); return e ? atoi(e) : 0; }();
  const int64_t sms = sm_count();
  const int64_t tiles = ceil_div(M, GM_BM) * ceil_div(N, GM_BN) * batch;
  // pairs pay off once the grid is saturated and there are at least two row tiles to pair
  const bool pair = force == 2 || (force == 0 && M > GM_BM && tiles >= 2 * sms);
  *cluster = pair ? 2 : 1;
  *width = 256;
  // under-filled grid: half-width tiles, quarter-width once even those leave half of the SMs idle
  if (!pair && narrow_ok && tiles < sms)
    *width = 2 * ceil_div(M, GM_BM) * ceil_div(N, 128) * batch <= sms ? 64 : 128;
}

int launch_gemm_tn(const GemmParams& p, cudaStream_t st) {
  MCLST_REQUIRE(p.M > 0 && p.N > 0 && p.nkb > 0 && (p.nseg == 1 || p.nseg == 3), MCLST_ERR_INVALID,
                "gemm: bad shape M=%lld N=%lld nkb=%d nseg=%d", (long long)p.M, (long long)p.N, p.nkb, p.nseg);
  MCLST_REQUIRE(p.nseg == 1 || (p.a_lo && p.b_lo), MCLST_ERR_INVALID, "gemm: split needs lo parts");
  MCLST_REQUIRE(p.c || p.lse_part, MCLST_ERR_INVALID, "gemm: neither an output nor statistics requested");
  MCLST_REQUIRE(p.a_nkb1 == 0 || (p.a_nkb1 > 0 && p.a_nkb1 <= p.nkb && p.batch <= 1 &&
                                  (p.a_nkb1 == p.nkb || (p.a2_hi && (p.nseg == 1 || p.a2_lo)))),
                MCLST_ERR_INVALID, "gemm: bad concatenated A operand");
  MCLST_REQUIRE(p.a1_mn == 0 || (p.a_nkb1 > 0 && p.a1_mn > 0), MCLST_ERR_INVALID, "gemm: transposed A needs a_nkb1");
  MCLST_REQUIRE(!p.lse_part || (!p.a_scale && !p.b_scale && !p.bias && p.act == 0 && p.batch <= 1),
                MCLST_ERR_INVALID, "gemm: the fused row statistics take a plain alpha-scaled product");
  GemmParams q = p;
  q.batch = std::max(1, p.batch);
  prof_mark(st, "gemm_tn");
  int cluster, width;
  // (the fused row statistics are laid out for 256-wide tiles)
  gemm_variant(p.M, p.N, q.batch, !p.lse_part && p.a_nkb1 == 0, &cluster, &width);
  if (cluster == 2) return launch_gemm_cl<2, 256>(q, st);
  if (width == 64) return launch_gemm_cl<1, 64>(q, st);
  if (width == 128) return launch_gemm_cl<1, 128>(q, st);
  return launch_gemm_cl<1, 256>(q, st);
}

// ---- operand bookkeeping --------------------------------------------------------------
size_t packed_operand_bytes(int64_t rows, int64_t k, bool is_b, int64_t* rows_pad, int* nkb) {
  const int64_t rp = (int64_t)align_up((size_t)rows, is_b ? GM_BN : GM_BM);
  const int kb = (int)ceil_div(k, TP_K);
  if (rows_pad) *rows_pad = rp;
  if (nkb) *nkb = kb;
  return (size_t)rp * kb * TP_K * 2;
}

PackedOperand take_operand(Arena& a, int64_t rows, int64_t k, bool is_b, bool split, int batch,
                           bool row_scaled) {
  PackedOperand o{};
  o.bytes = packed_operand_bytes(rows, k, is_b, &o.rows_pad, &o.nkb);
  o.hi = a.take<uint8_t>(o.bytes * batch);
  o.lo = split ? a.take<uint8_t>(o.bytes * batch) : nullptr;
  o.inv_scale = row_scaled ? a.take<float>((size_t)o.rows_pad * batch) : nullptr;
  return o;
}

}  // namespace mclst

using namespace mclst;

#ifdef GM_TIMING
extern "C" int mclst_debug_gemm_timing(unsigned long long* out, int n) {
  return (int)cudaMemcpyFromSymbol(out, mclst::g_gm_dbg, sizeof(unsigned long long) * (size_t)n);
}
#endif

// C-ABI: generic (batched) fp32 matmul through the split-precision tensor-core path -- the
// building block behind every nn.Linear / einsum on the path and their backward passes.
extern "C" int mclst_matmul_workspace_bytes(int64_t M, int64_t N, int64_t K, int batch, size_t* bytes) {
  MCLST_REQUIRE(bytes && M > 0 && N > 0 && K > 0 && batch >= 1, MCLST_ERR_INVALID,
                "matmul_workspace: bad args");
  Arena a(nullptr, 0);
  take_operand(a, M, K, false, true, batch, true);
  take_operand(a, N, K, true, true, batch, true);
  *bytes = align_up(a.off, 256);
  return 0;
}

extern "C" int mclst_debug_gemm_variant(int64_t M, int64_t N, int batch, int* cluster, int* width) {
  MCLST_REQUIRE(cluster && width && M > 0 && N > 0 && batch >= 1, MCLST_ERR_INVALID, "gemm_variant: bad args");
  gemm_variant(M, N, batch, true, cluster, width);
  return 0;
}

extern "C" int mclst_matmul(const float* A, int64_t lda, int a_trans, int64_t a_batch_stride,
                            const float* B, int64_t ldb, int b_trans, int64_t b_batch_stride,
                            float* C, int64_t ldc, int64_t c_batch_stride,
                            int64_t M, int64_t N, int64_t K, int batch, float alpha,
                            const float* bias, int act, const float* residual, int precise,
                            void* workspace, size_t workspace_bytes, mclst_stream_t stream) {
  MCLST_REQUIRE(A && B && C && workspace, MCLST_ERR_INVALID, "matmul: null pointer");
  MCLST_REQUIRE(M > 0 && N > 0 && K > 0 && batch >= 1, MCLST_ERR_INVALID, "matmul: bad shape");
  cudaStream_t st = (cudaStream_t)stream;
  // Two fp32-accurate routes.  The packed fp16 hi/lo path below pays a pack launch that reads and
  // writes both operands once before the product starts; the 3xTF32 kernel (gemm_tf32.cu) splits
  // inside the K loop, straight from the row-major tensors, at a lower MMA rate.  Measured inside
  // CUDA-graph replays on B200 (tools/gemm_bench.py, us: in-kernel split vs pack + product):
  //   [1024,256] x [256,256]^T            12.7 vs 18.4   short K: the pack is pure overhead
  //   [8,1024,1024] x [8,1024,64] (P V)   29.2 vs 45.7   a large batched operand used once
  //   [1024,1000] x [1000,1000]^T         28.0 vs 28.5   tie -> packed (fewer resident CTAs)
  //   [8,1024,64] x [8,1024,64]^T (Q K^T) 51.7 vs 36.9   output-bound: the packed path's epilogue
  const bool short_k = K <= 256 && (int64_t)M * N * batch <= (1 << 20);
  const bool batched_long = batch > 1 && K >= 512;
  if (precise && (short_k || batched_long) &&
      gemm_tf32x3_aligned(A, lda, a_trans, a_batch_stride, B, ldb, b_trans, b_batch_stride, K)) {
    const int rc = launch_gemm_tf32x3(A, lda, a_trans, a_batch_stride, B, ldb, b_trans, b_batch_stride, C, ldc,
                                      c_batch_stride, M, N, K, batch, alpha, bias, act, residual, st);
    prof_mark(st, "end");
    return rc;
  }
  Arena a(workspace, workspace_bytes);
  PackedOperand pa = take_operand(a, M, K, false, true, batch, true);
  PackedOperand pb = take_operand(a, N, K, true, true, batch, true);
  MCLST_REQUIRE(a.ok(), MCLST_ERR_WORKSPACE, "matmul: workspace too small");
  int rc;
  prof_mark(st, "pack_split");
  // a_trans: A is stored [K, M] (operand rows are its columns); likewise b_trans: B stored [K, N]
  if ((rc = launch_pack_pair(A, a_trans ? K : M, a_trans ? M : K, lda, a_trans != 0, pa, a_batch_stride,
                             B, b_trans ? K : N, b_trans ? N : K, ldb, b_trans != 0, pb, b_batch_stride,
                             batch, st))) return rc;
  GemmParams g{};
  g.a_hi = pa.hi; g.a_lo = pa.lo; g.b_hi = pb.hi; g.b_lo = pb.lo;
  g.a_batch_bytes = pa.bytes; g.b_batch_bytes = pb.bytes;
  g.a_scale = pa.inv_scale; g.b_scale = pb.inv_scale;
  g.a_scale_batch = (size_t)pa.rows_pad; g.b_scale_batch = (size_t)pb.rows_pad;
  g.nkb = pa.nkb; g.nseg = precise ? 3 : 1; g.M = M; g.N = N; g.c = C; g.ldc = ldc;
  g.c_batch_elems = (size_t)c_batch_stride;
  g.alpha = alpha; g.bias = bias; g.act = act; g.residual = residual; g.batch = batch;
  rc = launch_gemm_tn(g, st);
  prof_mark(st, "end");
  return rc;
}
