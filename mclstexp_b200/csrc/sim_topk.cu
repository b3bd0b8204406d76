// Cosine-similarity top-k on the 5th-generation tensor cores (find_matches,
// reference evel_her2st.py:74-84) -- candidate generation + exact re-rank.
//
//   pack_rows      fp32 rows -> L2-normalised fp16 "TilePack" operand (+ norm, fp16 rounding
//                  residual per row).  HBM-bound, one warp per row.
//   sim_topk       persistent-per-CTA GEMM: 128 queries (TMEM lanes) x 256 bank rows (TMEM
//                  columns) per tile, K <= 512.  Warp 0 streams bank slices with cp.async.bulk
//                  (TMA engine) into a 4-stage (K <= 256) or 3-stage (K <= 512) shared-memory
//                  ring, warp 1 issues
//                  tcgen05.mma.kind::f16 into a double-buffered 2 x 256-column TMEM
//                  accumulator, warps 2-9 drain it with tcgen05.ld: every thread owns one
//                  query row, compares 32 similarities per load against its running
//                  threshold and appends the rare survivors to a per-(query, stream) candidate
//                  buffer in global memory (L2 resident).  The Q x N similarity matrix is
//                  never materialised.
//   rerank         per query: merge the streams' candidates, keep those within 2*eps of the
//                  k-th best approximate score, recompute them exactly (fp64 accumulation of
//                  the fp32-normalised rows), sort by (value desc, index asc), emit top-k.
//
// Exactness argument (DESIGN.md "retrieval/exactness"): with |approx - exact| <= eps for
// every (query, row) pair -- eps = (r_q + max_s r_s) * (1 + 2^-9) + E_ACC, r = fp16 rounding
// residual norms measured at pack time (Cauchy-Schwarz), E_ACC the tensor-core accumulation
// bound (E_ACC_WIDE for K > 256) -- any row whose approximate score is below (k-th best approximate) - 2*eps is
// strictly worse than k rows, so it cannot be in the exact top-k.  The running threshold
// only ever uses a LOWER bound of the running k-th best, so nothing needed is dropped.
// Rows for which the band overflows the candidate buffer (massive ties, pathological
// clustering) are flagged and recomputed by the exact brute-force kernel.
#include <algorithm>
#include "common.cuh"
#include "retrieval.cuh"
#include "umma.cuh"

namespace mclst {

using namespace ptx;

// Bound on the tcgen05 fp32 accumulation error for |scores| <= 1, K <= 256.  Measured on
// B200 (tests/test_simtopk_gpu.py): max 1.5e-7 -- the bound keeps a 13x margin.
constexpr float E_ACC = 2.0e-6f;
// The same for 256 < K <= 512 (twice the accumulation steps, twice the bound).  Measured on B200
// (tests/test_retrieval_wide_gpu.py): max 2.3e-7 at K = 512 -- a 17x margin.  Each call carries
// the bound of its width (TcWorkspace::e_acc), so the bands and candidate counts of K <= 256 do
// not move.
constexpr float E_ACC_WIDE = 4.0e-6f;

// ============================================================================ pack_rows
// One warp per row (grid-stride).  CPL = 16-byte fp16 chunks per lane: 1 for dim <= 256 (lane l
// owns elements 8l..8l+7), 2 for dim <= 512 (chunks l and l + 32).  Per-row statistics are
// reduced per block before touching the global maximum: one atomic per row on a single address
// made the first version L2-atomic bound (1.3 ms for 1.06 M rows, 14 % of DRAM bandwidth).
template <bool VEC, int CPL>
__global__ void __launch_bounds__(256)
pack_rows_kernel(const float* __restrict__ x, int64_t rows, int64_t rows_pad, int64_t ld, int dim,
                 int nkb, uint8_t* __restrict__ packed, double* __restrict__ nrm,
                 float* __restrict__ resid, uint32_t* __restrict__ stats) {
  __shared__ uint32_t s_max[8];
  __shared__ uint32_t s_bad[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nchunks = nkb * 8;               // 16-byte chunks (8 halves) per row; <= 32 * CPL
  float run_max = 0.f;
  uint32_t run_bad = 0u;
  for (int64_t r = (int64_t)blockIdx.x * 8 + warp; r < rows_pad; r += (int64_t)gridDim.x * 8) {
    float v[8 * CPL];
#pragma unroll
    for (int i = 0; i < 8 * CPL; ++i) v[i] = 0.f;
#pragma unroll
    for (int c = 0; c < CPL; ++c) {
      const int chunk = lane + 32 * c;
      if (r < rows && chunk < nchunks) {
        const float* p = x + r * ld + chunk * 8;
        if (VEC) {                               // dim % 8 == 0, 16-byte aligned rows
          if (chunk * 8 < dim) {
            const float4 a = ldg_stream(reinterpret_cast<const float4*>(p));
            const float4 b = ldg_stream(reinterpret_cast<const float4*>(p) + 1);
            v[8 * c + 0] = a.x; v[8 * c + 1] = a.y; v[8 * c + 2] = a.z; v[8 * c + 3] = a.w;
            v[8 * c + 4] = b.x; v[8 * c + 5] = b.y; v[8 * c + 6] = b.z; v[8 * c + 7] = b.w;
          }
        } else {
#pragma unroll
          for (int i = 0; i < 8; ++i)
            if (chunk * 8 + i < dim) v[8 * c + i] = __ldg(p + i);
        }
      }
    }
    double ss = 0.0;
#pragma unroll
    for (int i = 0; i < 8 * CPL; ++i) ss = fma((double)v[i], (double)v[i], ss);
    ss = warp_sum(ss);
    const double n64 = fmax(sqrt(ss), 1e-12);
    // the fp16 operand only has to be an accurate normalisation (its rounding residual is
    // measured below and the 1e-6 slack of pair_eps covers the 2-ulp reciprocal)
    const float inv = (float)(1.0 / n64);
    float res = 0.f;
    uint32_t h2[4 * CPL];
#pragma unroll
    for (int i = 0; i < 4 * CPL; ++i) {
      const float a = v[2 * i] * inv, b = v[2 * i + 1] * inv;
      const __half ha = __float2half_rn(a), hb = __float2half_rn(b);
      const float da = a - __half2float(ha), db = b - __half2float(hb);
      res = fmaf(da, da, res);
      res = fmaf(db, db, res);
      h2[i] = (uint32_t)__half_as_ushort(ha) | ((uint32_t)__half_as_ushort(hb) << 16);
    }
    res = warp_sum(res);
#pragma unroll
    for (int c = 0; c < CPL; ++c) {
      const int chunk = lane + 32 * c;
      if (chunk < nchunks)
        *reinterpret_cast<uint4*>(packed + tilepack_chunk_offset(r, chunk, nkb)) =
            make_uint4(h2[4 * c], h2[4 * c + 1], h2[4 * c + 2], h2[4 * c + 3]);
    }
    if (lane == 0) {
      const float rr = (r < rows) ? sqrtf(res) * 1.00001f + 1e-12f : 0.f;
      nrm[r] = n64;
      resid[r] = rr;
      if (r < rows) {
        run_max = fmaxf(run_max, rr);
        if (!(ss <= 1.0e300)) run_bad = 1u;          // inf / NaN input
      }
    }
  }
  if (lane == 0) { s_max[warp] = __float_as_uint(run_max); s_bad[warp] = run_bad; }
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t m = 0u, bad = 0u;
    for (int w = 0; w < 8; ++w) { m = max(m, s_max[w]); bad |= s_bad[w]; }
    atomicMax(&stats[0], m);
    if (bad) atomicOr(&stats[1], 1u);
  }
}

// ============================================================================ sim_topk
constexpr int ST_STAGES = 4;
constexpr int ST_BN = 256;                      // bank rows per tile (TMEM columns)
constexpr int ST_STAGE_BYTES = 2 * TP_SLICE_BYTES;   // 256 rows x 64 halves
constexpr int ST_A_BYTES = 4 * TP_SLICE_BYTES;       // up to 4 K slices (dim <= 256)
// Wide variant (256 < dim <= 512): the resident query block takes 8 K slices (128 KiB), so the
// bank ring drops to 3 stages: 128 + 3 x 32 + 2 KiB = 231 424 B fits the 232 448 B opt-in limit,
// 4 stages would not.
constexpr int ST_STAGES_WIDE = 3;
constexpr int ST_A_BYTES_WIDE = 8 * TP_SLICE_BYTES;
static_assert(ST_A_BYTES_WIDE == TC_MAX_DIM / TP_K * TP_SLICE_BYTES, "resident query block of the widest rows");
constexpr int st_smem(int a_bytes, int stages) {
  return a_bytes + stages * ST_STAGE_BYTES + 1024 /*barriers*/ + 1024 /*align*/;
}
static_assert(st_smem(ST_A_BYTES_WIDE, ST_STAGES_WIDE) <= 232448, "wide sim_topk exceeds the shared-memory opt-in limit");
// Epilogue warps.  TMEM lanes can only be read by the warp whose id % 4 matches the lane quadrant,
// so two warps share a quadrant and split the 256 columns of a tile between them; each (query,
// column part) is its own candidate stream.  One epilogue warp per scheduler cannot hide its own
// dependent-issue latency (ncu on the 4-warp version: epilogue-bound at 25 % issue utilisation).
// Measured on B200, cfg4: 4 warps -> 34.7 ms, 8 -> 32.5 ms, 16 -> 36.4 ms (spills).
constexpr int ST_EPW = 8;
constexpr int ST_CP = ST_EPW / 4;               // column parts (candidate streams) per slot
constexpr int ST_THREADS = 64 + 32 * ST_EPW;
// At most 8 candidate streams per query (slots * ST_CP): the re-rank merges them in 16 KiB of
// shared memory per query.
constexpr int ST_MAX_SLOTS = 8 / ST_CP;

enum class SimPass {
  Candidates,   // the candidate pass: threshold filter into the per-(query, stream) buffers
  Seed,         // visit a strided sample of the bank tiles, record the maximum of every 32-score chunk
  Dump,         // testing aid: store the raw similarities
};

struct SimParams {
  const uint8_t* qpack;
  const uint8_t* bpack;
  int nkb;
  int64_t Q, N;
  int tiles_total, k;
  const float* q_resid;
  const uint32_t* bank_stats;
  uint2* cand;          // [q_pad][SS][CAP]  (approx score bits, bank row)
  int* cand_cnt;        // [q_pad][SS]       (-1: overflow, row goes to the exact path)
  uint32_t* gthr;       // [q_pad] running per-query threshold shared by all streams (ordered key, 0 = none)
  float* dump;          // Dump: raw similarities [Q, dump_ld]
  int64_t dump_ld;
  // Seed: visit n_tiles tiles tile_begin + i * tile_stride and only record the maximum of every
  // 32-score chunk into seed_out [q_pad][n_tiles * 8] (no candidates, no thresholds)
  float* seed_out;
  int tile_begin, tile_stride, n_tiles;
  float e_acc;          // accumulation bound of this width (pair_eps); sits in the tail padding
};

// eps: |tensor-core score - exact cosine| for a pair with fp16 residual norms rq, rs
// (Cauchy-Schwarz on the operand rounding) + accumulation bound e_acc of the call's width
// (E_ACC or E_ACC_WIDE) + fp32 normalisation slack.
__device__ __forceinline__ float pair_eps(float rq, float rs, float e_acc) {
  return 1.002f * (rq + rs) + e_acc + 1e-6f;
}

// Warp-cooperative prune of the candidate buffers of every lane with need == true:
// new threshold = (lower bound of the k-th best kept score) - e2; entries at or below it
// are dropped.  Leaves the buffer compacted in ascending bank index.  Deliberately NOT
// inlined: it runs once per ~10 tiles and inlining it 8x made the epilogue spill out of the
// instruction cache (ncu: 57% stall_no_inst in the first version).
struct PruneState { int cnt; float thr; int flagged; };

template <int CAP>
__device__ __noinline__ PruneState warp_prune(uint2* my_buf, uint32_t* my_gthr, int cnt, float thr,
                                              int flagged, bool need, int k, float e2) {
  constexpr int EPL = CAP / 32;
  const int lane = threadIdx.x & 31;
  unsigned mask = __ballot_sync(0xffffffffu, need);
  while (mask) {
    const int L = __ffs(mask) - 1;
    mask &= mask - 1;
    uint2* buf = reinterpret_cast<uint2*>(
        __shfl_sync(0xffffffffu, (unsigned long long)my_buf, L));
    const int n = __shfl_sync(0xffffffffu, cnt, L);
    const float le2 = __shfl_sync(0xffffffffu, e2, L);
    __syncwarp();
    uint32_t keys[EPL], vals[EPL], idxs[EPL];
#pragma unroll
    for (int j = 0; j < EPL; ++j) {
      const int i = lane + 32 * j;
      if (i < n) {
        const uint2 e = buf[i];
        vals[j] = e.x;
        idxs[j] = e.y;
        keys[j] = f2ord(__uint_as_float(e.x));
      } else {
        keys[j] = 0u; vals[j] = 0u; idxs[j] = 0u;
      }
    }
    // T = largest key with the low 8 bits clear such that at least k entries are >= T (greedy
    // bit descent).  The bits above the highest bit in which the smallest and the largest entry
    // differ are common to all entries -- the descent would pick them anyway -- so it starts
    // below them, and it settles two bits per step (three independent counts, one reduction
    // latency): ~8 dependent steps instead of 24.  The prune sits between tcgen05.ld and the
    // TMEM release of this warp, so its latency is what stalls the MMA pipe.
    uint32_t kmin = 0xffffffffu, kmax = 0u;
#pragma unroll
    for (int j = 0; j < EPL; ++j) {
      if (lane + 32 * j < n) { kmin = min(kmin, keys[j]); kmax = max(kmax, keys[j]); }
    }
    kmin = __reduce_min_sync(0xffffffffu, kmin);
    kmax = __reduce_max_sync(0xffffffffu, kmax);
    int bit = 31 - __clz((int)((kmin ^ kmax) | 0x100u));        // highest differing bit, >= 8
    uint32_t T = (bit >= 31) ? 0u : (kmax & ~((2u << bit) - 1u));
#pragma unroll 1
    for (; bit >= 9; bit -= 2) {
      const uint32_t c1 = T | (1u << (bit - 1)), c2 = T | (2u << (bit - 1)), c3 = T | (3u << (bit - 1));
      int n1 = 0, n2 = 0, n3 = 0;
#pragma unroll
      for (int j = 0; j < EPL; ++j) {
        n1 += (keys[j] >= c1) ? 1 : 0;
        n2 += (keys[j] >= c2) ? 1 : 0;
        n3 += (keys[j] >= c3) ? 1 : 0;
      }
      n1 = __reduce_add_sync(0xffffffffu, n1);
      n2 = __reduce_add_sync(0xffffffffu, n2);
      n3 = __reduce_add_sync(0xffffffffu, n3);
      T = (n3 >= k) ? c3 : (n2 >= k) ? c2 : (n1 >= k) ? c1 : T;
    }
    if (bit == 8) {
      const uint32_t cand = T | (1u << 8);
      int c = 0;
#pragma unroll
      for (int j = 0; j < EPL; ++j) c += (keys[j] >= cand) ? 1 : 0;
      c = __reduce_add_sync(0xffffffffu, c);
      if (c >= k) T = cand;
    }
    // T <= key of the k-th best (low 8 bits cleared): conservative lower bound.  Publish it
    // and adopt whatever better bound another stream of the same query already found.
    // (published fire-and-forget: every stream of this query adopts it at its next tile, and
    // the prune never waits on an L2 round trip)
    const float new_thr = ord2f(T) - le2;
    if (lane == L) atomicMax(my_gthr, f2ord(new_thr));
    int out = 0;
#pragma unroll
    for (int j = 0; j < EPL; ++j) {
      const int i = lane + 32 * j;
      const bool keep = (i < n) && (__uint_as_float(vals[j]) > new_thr);
      const unsigned bal = __ballot_sync(0xffffffffu, keep);
      if (keep) buf[out + __popc(bal & ((1u << lane) - 1u))] = make_uint2(vals[j], idxs[j]);
      out += __popc(bal);
    }
    __syncwarp();
    if (lane == L) {
      cnt = out;
      thr = new_thr;
      if (out > CAP - 64) {            // band denser than the buffer: give the row to the exact path
        flagged = 1;
        thr = __int_as_float(0x7f800000);
      }
    }
  }
  PruneState r;
  r.cnt = cnt; r.thr = thr; r.flagged = flagged;
  return r;
}

// One 32-column chunk of one query row: append every similarity above the running threshold.
// Two-level test (chunk max, then FILTER_GS-wide group max) keeps the common "one survivor in
// the warp" case short; the bank-tail bound check lives in a separate (cold) instantiation.
// Groups of 4 and 16 were measured too (DESIGN.md §3).
constexpr int FILTER_GS = 8;
template <int CAP, bool TAIL>
__device__ __forceinline__ void filter_groups(const uint32_t (&v)[32], const float (&g)[32 / FILTER_GS],
                                              uint2* my_buf, int& cnt, float thr, uint32_t nb,
                                              int n_left) {
#pragma unroll
  for (int h = 0; h < 32 / FILTER_GS; ++h) {
    if (g[h] > thr) {
#pragma unroll
      for (int j = 0; j < FILTER_GS; ++j) {
        const int e = FILTER_GS * h + j;
        if (__uint_as_float(v[e]) > thr && (!TAIL || e < n_left))
          my_buf[cnt++] = make_uint2(v[e], nb + e);
      }
    }
  }
}

template <int CAP>
__device__ __forceinline__ void filter_chunk(const uint32_t (&v)[32], uint2* my_buf,
                                             uint32_t* my_gthr, int& cnt, float& thr, int& flagged,
                                             uint32_t nb, int n_left, int k, float e2) {
  constexpr int NG = 32 / FILTER_GS;
  float g[NG];
#pragma unroll
  for (int h = 0; h < NG; ++h) {
    float m = __uint_as_float(v[FILTER_GS * h]);
#pragma unroll
    for (int j = 1; j < FILTER_GS; ++j) m = fmaxf(m, __uint_as_float(v[FILTER_GS * h + j]));
    g[h] = m;
  }
  float mall = g[0];
#pragma unroll
  for (int h = 1; h < NG; ++h) mall = fmaxf(mall, g[h]);
  if (mall > thr) {
    if (n_left >= 32) filter_groups<CAP, false>(v, g, my_buf, cnt, thr, nb, n_left);
    else filter_groups<CAP, true>(v, g, my_buf, cnt, thr, nb, n_left);
  }
  // prune when the buffer cannot take another full chunk.  (Earlier prunes, every few appended
  // entries, tighten the threshold sooner but were measured slower while thresholds converge.)
  const bool need = cnt > CAP - 32;
  if (__any_sync(0xffffffffu, need)) {
    const PruneState ps = warp_prune<CAP>(my_buf, my_gthr, cnt, thr, flagged, need, k, e2);
    cnt = ps.cnt; thr = ps.thr; flagged = ps.flagged;
  }
}

// ============================================================================ sim_topk (lanes)
// Persistent: one CTA ("lane") per SM walks a short list of units (query block, bank-tile range,
// candidate slot), so that every SM gets the same number of tiles whatever the number of query
// blocks.  A (query block x stream) grid idles SMs whenever blocks * streams is not close to a
// multiple of 148 (128 blocks on 148 SMs: 14 % lost, which is what the 4x2 eight-GPU decomposition
// ran into) and pays for balance with extra streams per query (4 at 256 blocks: twice the
// candidates for the re-rank).  Unit lists, QT blocks, T tiles, W lanes (LanePlan, retrieval.cuh):
//   * rounds = QT / W full rounds: lane c takes block j*W + c over the whole bank (slot 0);
//   * the rest = QT % W blocks share one last round of rest*T/W tiles per lane: each block gets
//     w = W / rest dedicated lanes that split the MAIN region [0, M) of the bank w ways
//     (slots 0..w-1), and the R = W - w*rest left-over lanes cut the TAIL region [M, T) of all
//     rest blocks into equal linear runs (slots w, w+1), M = T*w*rest/W.
// Lanes of a round start together and advance at the same rate, so all of them read the same
// bank tiles at about the same time (one HBM read, the rest L2 hits); tail lanes take their
// boundary-aligned pieces first and the partial head piece last for the same reason (two aligned
// groups instead of R unrelated streams).
struct LaneUnit { int qb, t0, t1, slot; };

__host__ __device__ inline bool lane_unit(const LanePlan& L, int T, int c, int j, LaneUnit& u) {
  if (j < L.rounds * L.h) {
    const int r = j / L.h, sub = j - r * L.h;
    u.qb = r * L.W + c;
    u.t0 = (int)((int64_t)T * sub / L.h);
    u.t1 = (int)((int64_t)T * (sub + 1) / L.h);
    u.slot = sub;
    return true;
  }
  j -= L.rounds * L.h;
  if (L.rest == 0) return false;
  const int main_lanes = L.w * L.rest;
  if (c < main_lanes) {
    if (j >= L.hm) return false;
    const int ql = c / L.w, part = (c - ql * L.w) * L.hm + j, parts = L.w * L.hm;
    u.qb = L.rounds * L.W + ql;
    u.t0 = (int)((int64_t)L.M * part / parts);
    u.t1 = (int)((int64_t)L.M * (part + 1) / parts);
    u.slot = part;
    return true;
  }
  if (c >= main_lanes + L.R) return false;
  const int64_t Tt = T - L.M;
  const int jt = c - main_lanes;
  const int64_t lo = (int64_t)jt * L.Lt;
  const int64_t end = (int64_t)L.rest * Tt;
  const int64_t hi = lo + L.Lt < end ? lo + L.Lt : end;
  if (lo >= hi) return false;
  const int64_t first_b = (lo + Tt - 1) / Tt * Tt;                    // first block boundary >= lo
  const int64_t head_end = first_b < hi ? first_b : hi;              // head piece = [lo, head_end)
  const int64_t nb = hi > first_b ? (hi - first_b + Tt - 1) / Tt : 0;  // boundary-aligned pieces
  int64_t a, b;
  if (j < nb) { a = first_b + (int64_t)j * Tt; b = a + Tt < hi ? a + Tt : hi; }
  else if (j == nb && head_end > lo) { a = lo; b = head_end; }
  else return false;
  const int64_t ql = a / Tt;
  u.qb = L.rounds * L.W + (int)ql;
  u.t0 = L.M + (int)(a - ql * Tt);
  u.t1 = L.M + (int)(b - ql * Tt);
  u.slot = L.w * L.hm + jt - (int)((ql * Tt) / L.Lt);
  return true;
}

static LanePlan plan_lanes(int64_t qt, int64_t T, int W, int max_slots) {
  LanePlan L{};
  L.W = (int)std::min<int64_t>(W, std::max<int64_t>(qt, 1) * max_slots);
  L.W = std::max(1, std::min(L.W, W));
  L.rounds = (int)(qt / L.W);
  L.rest = (int)(qt % L.W);
  L.w = 0; L.R = 0; L.M = (int)T; L.Lt = 0; L.slots = 1;
  if (L.rest > 0) {
    int w = L.W / L.rest;
    w = (int)std::min<int64_t>(std::min(w, max_slots), std::max<int64_t>(T, 1));
    L.w = std::max(1, w);
    const int left = L.W - L.w * L.rest;
    if (left > 0 && left < L.rest && L.w + 2 <= max_slots) {
      // main region length: whichever rounding of T*w*rest/W gives the smaller makespan
      const int64_t m_lo = T * L.w * L.rest / L.W;
      int64_t best_m = T, best_span = ceil_div(T, (int64_t)L.w);
      for (int64_t M = m_lo; M <= std::min(T - 1, m_lo + 1); ++M) {
        if (M < L.w) continue;
        const int64_t span = std::max(ceil_div(M, (int64_t)L.w), ceil_div((int64_t)L.rest * (T - M), (int64_t)left));
        if (span < best_span) { best_span = span; best_m = M; }
      }
      if (best_m < T) {
        L.R = left; L.M = (int)best_m;
        L.Lt = (int)ceil_div((int64_t)L.rest * (T - best_m), (int64_t)left);
      }
    }
    L.slots = L.w + (L.R > 0 ? 2 : 0);
  }
  // Fresh candidate buffers instead of prunes: a unit cut into h back-to-back sub-units gives each
  // its own slot, so the later ones start from the threshold the earlier ones published and rarely
  // fill up (one long stream per query block cost 2 ms of extra prune stalls at cfg4).
  constexpr int split = 2;
  L.h = (int)std::max<int64_t>(1, std::min<int64_t>(std::min(split, max_slots), T));
  L.hm = 1;
  if (L.rest > 0) {
    const int room = (max_slots - (L.R > 0 ? 2 : 0)) / L.w;
    L.hm = (int)std::max<int64_t>(1, std::min<int64_t>(std::min(split, room), std::max<int64_t>(1, L.M / L.w)));
    L.slots = L.w * L.hm + (L.R > 0 ? 2 : 0);
  }
  if (L.rounds > 0) L.slots = std::max(L.slots, L.h);
  return L;
}

// PASS (SimPass) selects what the epilogue does with the scores of a tile.  In the Seed pass
// "tile" t of a unit is bank tile tile_begin + t * tile_stride of the sample.  A_BYTES (resident
// query block) and STAGES (bank ring) are ST_A_BYTES / ST_STAGES for dim <= 256 and
// ST_A_BYTES_WIDE / ST_STAGES_WIDE for dim <= 512; nothing else depends on the width.
template <int CAP, SimPass PASS, int A_BYTES, int STAGES>
__global__ void __launch_bounds__(ST_THREADS, 1)
sim_topk_lanes_kernel(const SimParams p, const LanePlan L) {
  constexpr bool SEED = PASS == SimPass::Seed;
  constexpr int PART_COLS = ST_BN / ST_CP;
  constexpr int NCH = PART_COLS / 32;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = smem;
  uint8_t* sB = smem + A_BYTES;
  uint64_t* bar_full = reinterpret_cast<uint64_t*>(sB + STAGES * ST_STAGE_BYTES);
  uint64_t* bar_empty = bar_full + STAGES;
  uint64_t* bar_a = bar_empty + STAGES;
  uint64_t* bar_afree = bar_a + 1;
  uint64_t* bar_tfull = bar_afree + 1;
  uint64_t* bar_tempty = bar_tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_tempty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = blockIdx.x;
  const int nkb = p.nkb;
  const int T = SEED ? p.n_tiles : p.tiles_total;

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&bar_full[i], 1); mbar_init(&bar_empty[i], 1); }
    mbar_init(bar_a, 1);
    mbar_init(bar_afree, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(&bar_tfull[i], 1); mbar_init(&bar_tempty[i], ST_EPW); }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    // Every CTA fetches its own bank slices: multicasting them across a cluster of CTAs that stream
    // the same tiles was correct but slower on B200 (cfg4) -- L2 -> SM traffic is not the limiter.
    if (lane == 0) {
      const uint64_t pol_keep = policy_evict_last();
      uint32_t stage = 0, phase = 0;
      LaneUnit u;
      for (int j = 0; lane_unit(L, T, c, j, u); ++j) {
        if (j > 0) mbar_wait(bar_afree, (uint32_t)(j - 1) & 1u);   // previous unit's MMAs have read sA
        mbar_arrive_expect_tx(bar_a, (uint32_t)(nkb * TP_SLICE_BYTES));
        for (int kb = 0; kb < nkb; ++kb)
          bulk_g2s(sA + kb * TP_SLICE_BYTES,
                   p.qpack + ((size_t)u.qb * nkb + kb) * TP_SLICE_BYTES, TP_SLICE_BYTES, bar_a);
        for (int t = u.t0; t < u.t1; ++t) {
          const int bt = SEED ? p.tile_begin + t * p.tile_stride : t;       // bank tile
          for (int kb = 0; kb < nkb; ++kb) {
            mbar_wait(&bar_empty[stage], phase ^ 1);
            mbar_arrive_expect_tx(&bar_full[stage], ST_STAGE_BYTES);
            uint8_t* dst = sB + stage * ST_STAGE_BYTES;
            bulk_g2s_hint(dst, p.bpack + ((size_t)(2 * bt) * nkb + kb) * TP_SLICE_BYTES, TP_SLICE_BYTES,
                          &bar_full[stage], pol_keep);
            bulk_g2s_hint(dst + TP_SLICE_BYTES, p.bpack + ((size_t)(2 * bt + 1) * nkb + kb) * TP_SLICE_BYTES,
                          TP_SLICE_BYTES, &bar_full[stage], pol_keep);
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    // the whole warp walks the loop (uniform control flow: descriptors in uniform registers), one
    // elected lane issues -- umma.cuh: elect_one
    constexpr uint32_t idesc = make_idesc_f16(128, ST_BN, false);
    const uint32_t leader = elect_one();
    const uint32_t a_base = smem_u32(sA);
    const uint32_t b_base = smem_u32(sB);
    uint32_t stage = 0, phase = 0;
    int it = 0;
    LaneUnit u;
    for (int j = 0; lane_unit(L, T, c, j, u); ++j) {
      mbar_wait(bar_a, (uint32_t)j & 1u);
      tc_fence_after();
      for (int t = u.t0; t < u.t1; ++t, ++it) {
        const int buf = it & 1;
        mbar_wait(&bar_tempty[buf], ((it >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * ST_BN;
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&bar_full[stage], phase);
          tc_fence_after();
          if (leader) {
#pragma unroll
            for (int k4 = 0; k4 < 4; ++k4) {
              const uint64_t ad = make_smem_desc_sw128(a_base + kb * TP_SLICE_BYTES + k4 * 32);
              const uint64_t bd = make_smem_desc_sw128(b_base + stage * ST_STAGE_BYTES + k4 * 32);
              mma_f16_ss(d_tmem, ad, bd, idesc, (kb | k4) != 0 ? 1u : 0u);
            }
            mma_commit(&bar_empty[stage]);
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        if (leader) mma_commit(&bar_tfull[buf]);
        __syncwarp();
      }
      if (leader) mma_commit(bar_afree);
      __syncwarp();
    }
  } else {
    // ------------------------------------------------------------ epilogue: threshold filter
    // The filter runs on the warps that read TMEM.  Handing passing chunks to separate worker
    // warps through a shared-memory event ring was bit-exact and 2 % faster once thresholds are
    // warm (26.1 vs 26.7 ms at cfg4), but the workers fell behind while thresholds converge (38 vs
    // 32 ms end to end).
    const int quad = warp & 3;
    const int part = (warp - 2) >> 2;
    const int row = quad * 32 + lane;
    const int SS = L.slots * ST_CP;
    const float rs_max = __uint_as_float(p.bank_stats[0]);
    const int k = p.k;
    const uint32_t t_lane = tmem_base + ((uint32_t)(quad * 32) << 16) + part * PART_COLS;
    int it = 0;
    LaneUnit u;
#pragma unroll 1
    for (int j = 0; lane_unit(L, T, c, j, u); ++j) {
      const int64_t q = (int64_t)u.qb * 128 + row;
      const bool q_valid = q < p.Q;
      const int stream = u.slot * ST_CP + part;
      uint2* my_buf = p.cand + ((size_t)q * SS + stream) * CAP;
      uint32_t* my_gthr = p.gthr + q;
      const float rq = q_valid ? p.q_resid[q] : 0.f;
      const float e2 = 2.02f * pair_eps(rq, rs_max, p.e_acc);
      float thr = q_valid ? __int_as_float(0xff800000) : __int_as_float(0x7f800000);
      int cnt = 0;
      int flagged = 0;
#pragma unroll 1
      for (int t = u.t0; t < u.t1; ++t, ++it) {
        const int buf = it & 1;
        // adopt the best threshold any other stream of this query has published so far
        const uint32_t gk = q_valid ? *reinterpret_cast<volatile uint32_t*>(my_gthr) : 0u;
        mbar_wait(&bar_tfull[buf], (it >> 1) & 1);
        tc_fence_after();
        if (gk != 0u) thr = fmaxf(thr, ord2f(gk));
        const uint32_t taddr = t_lane + buf * ST_BN;
        const int64_t col_base = (int64_t)(SEED ? p.tile_begin + t * p.tile_stride : t) * ST_BN + part * PART_COLS;
        const int n_valid = (int)min((int64_t)PART_COLS, p.N - col_base);
        uint32_t va[32], vb[32];
        if constexpr (PASS != SimPass::Candidates) {
          // Seed: the maximum of every 32-score chunk of this thread's columns; Dump: the scores
          float* out = SEED ? p.seed_out + (size_t)q * (p.n_tiles * 8) + (size_t)t * 8 + part * NCH
                            : p.dump + q * p.dump_ld + col_base;
#pragma unroll 1
          for (int ch = 0; ch < NCH; ++ch) {
            tmem_ld_32x32(taddr + ch * 32, va);
            tmem_ld_wait();
            if constexpr (SEED) {
              float m = -INFINITY;
#pragma unroll
              for (int e = 0; e < 32; ++e)
                m = fmaxf(m, (ch * 32 + e < n_valid) ? __uint_as_float(va[e]) : -INFINITY);
              if (q_valid) out[ch] = m;
            } else if (q_valid) {
#pragma unroll
              for (int e = 0; e < 32; ++e)
                if (ch * 32 + e < n_valid) out[ch * 32 + e] = __uint_as_float(va[e]);
            }
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&bar_tempty[buf]);
          continue;
        }
        tmem_ld_32x32(taddr, va);
#pragma unroll 1
        for (int ch = 0; ch < NCH; ch += 2) {
          tmem_ld_wait();
          tmem_ld_32x32(taddr + (ch + 1) * 32, vb);
          filter_chunk<CAP>(va, my_buf, my_gthr, cnt, thr, flagged, (uint32_t)(col_base + ch * 32),
                            n_valid - ch * 32, k, e2);
          tmem_ld_wait();
          if (ch + 2 < NCH) {
            tmem_ld_32x32(taddr + (ch + 2) * 32, va);
          } else {
            // this warp's columns are in registers: hand the accumulator back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar_tempty[buf]);
          }
          filter_chunk<CAP>(vb, my_buf, my_gthr, cnt, thr, flagged,
                            (uint32_t)(col_base + (ch + 1) * 32), n_valid - (ch + 1) * 32, k, e2);
        }
      }
      if (PASS == SimPass::Candidates && q_valid) p.cand_cnt[(size_t)q * SS + stream] = flagged ? -1 : cnt;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// ============================================================================ seed thresholds
// gthr[q] = (24-bit lower bound of the k-th largest chunk maximum of the sample) - e2.  The k
// largest chunk maxima are k distinct bank rows, so this is a valid lower bound of the k-th
// best score of the whole bank, minus the band: every stream starts warm instead of with -inf.
__global__ void __launch_bounds__(128)
seed_threshold_kernel(const float* __restrict__ seed, int n_vals, int64_t Q, int k,
                      const float* __restrict__ q_resid, const uint32_t* __restrict__ bank_stats,
                      uint32_t* __restrict__ gthr, int k2, float* __restrict__ bound_k,
                      float* __restrict__ bound_part, float* __restrict__ spec_out, float e_acc) {
  // k < top_k is the SPECULATIVE start (see spec_rank): the threshold is then only valid if fewer
  // than k of the true top rows fell into the sample; spec_out records it so that the re-rank can
  // verify the outcome with one compare (and send the query to the exact path otherwise).
  const int lane = threadIdx.x & 31;
  const int64_t q = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
  if (q >= Q) return;
  const float* v = seed + (size_t)q * n_vals;
  uint32_t T = 0, T2 = 0;       // T2: the k2-th largest (k2 <= k), for the cross-shard bound
  if (n_vals <= 1024) {
    // the usual case: the whole sample as ordered keys in registers, 24 compare sweeps
    uint32_t key[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) key[i] = (lane + 32 * i < n_vals) ? f2ord(v[lane + 32 * i]) : 0u;
    for (int bit = 31; bit >= 8; --bit) {
      const uint32_t cand = T | (1u << bit);
      int c = 0;
#pragma unroll
      for (int i = 0; i < 32; ++i) c += (key[i] >= cand) ? 1 : 0;
      c = __reduce_add_sync(0xffffffffu, c);
      if (c >= k) T = cand;
    }
    if (bound_part) {
      for (int bit = 31; bit >= 8; --bit) {
        const uint32_t cand = T2 | (1u << bit);
        int c = 0;
#pragma unroll
        for (int i = 0; i < 32; ++i) c += (key[i] >= cand) ? 1 : 0;
        c = __reduce_add_sync(0xffffffffu, c);
        if (c >= k2) T2 = cand;
      }
    }
  } else {
    for (int bit = 31; bit >= 8; --bit) {
      const uint32_t cand = T | (1u << bit);
      int c = 0;
      for (int i = lane; i < n_vals; i += 32) c += (f2ord(v[i]) >= cand) ? 1 : 0;
      c = __reduce_add_sync(0xffffffffu, c);
      if (c >= k) T = cand;
    }
    if (bound_part) {
      for (int bit = 31; bit >= 8; --bit) {
        const uint32_t cand = T2 | (1u << bit);
        int c = 0;
        for (int i = lane; i < n_vals; i += 32) c += (f2ord(v[i]) >= cand) ? 1 : 0;
        c = __reduce_add_sync(0xffffffffu, c);
        if (c >= k2) T2 = cand;
      }
    }
  }
  if (lane == 0) {
    const float e1 = 1.01f * pair_eps(q_resid[q], __uint_as_float(bank_stats[0]), e_acc);
    float spec = -INFINITY;
    if (T != 0u) {
      const float thr = ord2f(T) - 2.f * e1;
      if (thr == thr && thr > -INFINITY) { gthr[q] = f2ord(thr); spec = thr; }
    }
    if (spec_out) spec_out[q] = spec;
    // lower bounds of EXACT scores: at least k (k2) rows of this shard score >= bound
    if (bound_k) { const float b = ord2f(T) - e1; bound_k[q] = (T != 0u && b == b) ? b : -INFINITY; }
    if (bound_part) { const float b = ord2f(T2) - e1; bound_part[q] = (T2 != 0u && b == b) ? b : -INFINITY; }
  }
}

// After the candidate pass: a lower bound of this shard's exact k-th best score per query, for the
// exchange between bank shards before their re-ranks.  Taken from the candidates themselves: the
// k-th largest tensor-core score among everything the streams kept (radix descent over the keys,
// held in shared memory), minus eps.  The running threshold alone is not enough -- a stream only
// tightens it when its buffer fills, which a small shard with a good seed never does.
constexpr int KB_MAX = 2048;      // candidates examined per query (more: fall back to the threshold)
__global__ void __launch_bounds__(128)
export_bound_kernel(const uint2* __restrict__ cand, const int* __restrict__ cand_cnt, int SS, int cap, int k,
                    const uint32_t* __restrict__ gthr, int64_t Q, const float* __restrict__ q_resid,
                    const uint32_t* __restrict__ bank_stats, float* __restrict__ bound, int k_part,
                    float* __restrict__ bound_part, float e_acc) {
  __shared__ uint32_t keys[4][KB_MAX];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t q = (int64_t)blockIdx.x * 4 + warp;
  if (q >= Q) return;
  const float e1 = 1.01f * pair_eps(q_resid[q], __uint_as_float(bank_stats[0]), e_acc);
  float b = -INFINITY;
  const uint32_t gk = gthr[q];
  if (gk != 0u) {                      // threshold = (lower bound of the k-th best score) - 2.02 eps
    const float v = ord2f(gk) + e1;
    if (v == v && v < INFINITY) b = v;
  }
  int M = 0;
  bool ok = true;
  for (int s = 0; s < SS && ok; ++s) {
    const int c = cand_cnt[(size_t)q * SS + s];
    if (c < 0 || M + c > KB_MAX) { ok = false; break; }
    const uint2* src = cand + ((size_t)q * SS + s) * cap;
    for (int i = lane; i < c; i += 32) keys[warp][M + i] = f2ord(__uint_as_float(src[i].x));
    M += c;
  }
  __syncwarp();
  if (ok && M >= k) {
    uint32_t T = 0;
    for (int bit = 31; bit >= 8; --bit) {
      const uint32_t candT = T | (1u << bit);
      int c = 0;
      for (int i = lane; i < M; i += 32) c += (keys[warp][i] >= candT) ? 1 : 0;
      c = __reduce_add_sync(0xffffffffu, c);
      if (c >= k) T = candT;
    }
    const float v = ord2f(T) - e1;
    if (T != 0u && v == v && v < INFINITY) b = fmaxf(b, v);
  }
  // the k_part-th best of this shard (k_part = ceil(k / shards)): the MINIMUM of these over the
  // shards bounds the global k-th best too, and for shards of similar content it sits at global
  // rank ~k instead of ~k * shards
  float bp = b;
  if (bound_part && ok && M >= k_part) {
    uint32_t T = 0;
    for (int bit = 31; bit >= 8; --bit) {
      const uint32_t candT = T | (1u << bit);
      int c = 0;
      for (int i = lane; i < M; i += 32) c += (keys[warp][i] >= candT) ? 1 : 0;
      c = __reduce_add_sync(0xffffffffu, c);
      if (c >= k_part) T = candT;
    }
    const float v = ord2f(T) - e1;
    if (T != 0u && v == v && v < INFINITY) bp = fmaxf(bp, v);
  }
  if (lane == 0) {
    bound[q] = b;
    if (bound_part) bound_part[q] = bp;
  }
}

__global__ void fill_kernel(float* __restrict__ x, int64_t n, float v) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] = v;
}

// Cross-shard warm start: `bound` is a lower bound of the exact GLOBAL k-th best score of every
// query (exchanged between the ranks that hold the other bank shards).  A row of this shard whose
// tensor-core score is below bound - 1.01 eps is strictly worse than k rows somewhere, so the
// running threshold may start there.
__global__ void __launch_bounds__(256)
apply_bound_kernel(const float* __restrict__ bound, int64_t Q, const float* __restrict__ q_resid,
                   const uint32_t* __restrict__ bank_stats, uint32_t* __restrict__ gthr, float e_acc) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= Q) return;
  const float b = bound[q];
  if (!(b > -INFINITY) || !(b < INFINITY)) return;
  const float thr = b - 1.01f * pair_eps(q_resid[q], __uint_as_float(bank_stats[0]), e_acc);
  if (thr == thr && thr > -INFINITY) {
    const uint32_t key = f2ord(thr);
    if (key > gthr[q]) gthr[q] = key;
  }
}

// ============================================================================ rerank
constexpr int RR_MAX = 512;      // most survivors re-ranked exactly per query (more -> exact path)

struct RerankParams {
  const uint2* cand;
  const int* cand_cnt;
  int SS, cap, k;               // SS = candidate streams per query
  int64_t Q, N;
  const float* bank; int64_t ldb; const double* bank_nrm;
  const float* query; int64_t ldq; const double* q_nrm; const float* q_resid;
  const uint32_t* bank_stats; const uint32_t* q_stats;
  const uint32_t* gthr;            // final shared threshold per query (valid lower bound of the band)
  int dim;
  int64_t index_offset;
  int64_t* out_idx; float* out_val;
  float* out_dist; int dist_p;     // optional: L1 (p=1) / L2 (p=2) distance of each winner to the raw query
  int* fb_list; int* counters;     // counters[0] = fallback count, [1] = resolved here
  int allow_partial;               // an external bound was applied: fewer than k survivors is legitimate
  float e_acc;                     // accumulation bound of this width (pair_eps); sits in padding
  const float* spec;               // speculative start threshold per query (NaN / -inf: none)
};

// exact cosine of one bank row against the query held in qh[] (raw values as doubles):
// fp64 dot of the raw fp32 rows / (fp64 norm product), rounded once to fp32.  VPL values per
// lane: 8 for dim <= 256, 16 for dim <= 512.
template <bool VEC, bool L1, int VPL>
__device__ __forceinline__ double row_dot(const float* __restrict__ sp, const double (&qh)[VPL],
                                          int dim, int lane, float* l1) {
  double acc = 0.0;
  float v[VPL];
  if (VEC) {                       // dim == 8 * VPL, 16-byte aligned rows: d = 4*lane + 128*h + i
#pragma unroll
    for (int h = 0; h < VPL / 4; ++h) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(sp) + 32 * h + lane);
      v[4 * h] = a.x; v[4 * h + 1] = a.y; v[4 * h + 2] = a.z; v[4 * h + 3] = a.w;
    }
  } else {                         // d = lane + 32*t
#pragma unroll
    for (int t = 0; t < VPL; ++t) {
      const int d = lane + 32 * t;
      v[t] = d < dim ? __ldg(sp + d) : 0.f;
    }
  }
#pragma unroll
  for (int t = 0; t < VPL; ++t) acc = fma((double)v[t], qh[t], acc);
  if (L1) {                        // (compile-time: predicated off it still cost 10 % of the kernel's issue slots)
    float s = 0.f;
#pragma unroll
    for (int t = 0; t < VPL; ++t) s += fabsf(v[t] - (float)qh[t]);
    *l1 = s;
  }
  return acc;
}

constexpr int RR_MIN_BLOCKS = 4;   // 5 (96 registers, 140 B of spills) measured equal: latency is hidden by the 4x unrolled loads
// VPL = query values per lane (8: dim <= 256, 16: dim <= 512).  The gather keeps the bytes in
// flight per warp rather than the row count: 8 rows of 1 KiB or 4 rows of 2 KiB (16 values x 8
// rows would take 128 registers for the loads alone).
template <bool VEC, bool WANT_L1, int VPL>
__global__ void __launch_bounds__(128, RR_MIN_BLOCKS)
rerank_kernel(const RerankParams p, int warps_per_block, int per_warp_entries) {
  constexpr int RPI = 64 / VPL;              // rows gathered per step
  extern __shared__ __align__(16) unsigned char rr_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t q = (int64_t)blockIdx.x * warps_per_block + warp;
  if (warp >= warps_per_block || q >= p.Q) return;
  unsigned long long* ent = reinterpret_cast<unsigned long long*>(rr_smem) +
                            (size_t)warp * per_warp_entries;   // (key << 32) | idx, later sort keys
  // distance payload of the survivors + the permutation the sort applies to them
  float* pay = reinterpret_cast<float*>(reinterpret_cast<unsigned long long*>(rr_smem) +
                                        (size_t)warps_per_block * per_warp_entries) + (size_t)warp * RR_MAX;
  unsigned short* slot = reinterpret_cast<unsigned short*>(
      reinterpret_cast<float*>(reinterpret_cast<unsigned long long*>(rr_smem) +
                               (size_t)warps_per_block * per_warp_entries) + (size_t)warps_per_block * RR_MAX) +
      (size_t)warp * RR_MAX;
  const bool want_dist = p.out_dist != nullptr;
  constexpr bool want_l1 = WANT_L1;          // (host: out_dist != nullptr && dist_p == 1)
  // ---- gather the streams' candidates
  bool bad = (p.bank_stats[1] | p.q_stats[1]) != 0;    // non-finite input: exact path decides
  int M = 0;
  // Every stream dropped only scores at or below a threshold that was <= the final shared one,
  // and the shared one is itself <= (k-th best) - 2 eps: stale entries below it go right away.
  // If the buffer still fills up, the band is tightened from what has been gathered so far
  // (the k-th best of any subset is a lower bound of the global k-th best) and gathering resumes.
  uint32_t g_key = p.gthr[q];
  const float rs_max = __uint_as_float(p.bank_stats[0]);
  const float e2 = 2.02f * pair_eps(p.q_resid[q], rs_max, p.e_acc);
  auto tighten = [&](int count) -> int {      // radix descent (24 bits) + in-place band compaction
    // the keys are cosines of one narrow range: their leading bits agree (typically 9-10 of them),
    // and the descent starts below that common prefix instead of confirming it bit by bit
    uint32_t k_and = 0xffffffffu, k_or = 0u;
    for (int i = lane; i < count; i += 32) { const uint32_t kk = (uint32_t)(ent[i] >> 32); k_and &= kk; k_or |= kk; }
    k_and = __reduce_and_sync(0xffffffffu, k_and);
    k_or = __reduce_or_sync(0xffffffffu, k_or);
    const uint32_t diff = (k_and ^ k_or) & 0xffffff00u;
    const int top = diff ? 31 - __clz(diff) : 7;          // highest bit (>= 8) on which two keys differ
    uint32_t T = (top < 31) ? (k_and & ~((2u << top) - 1u)) : 0u;
    for (int bit = top; bit >= 8; --bit) {
      const uint32_t candT = T | (1u << bit);
      int c = 0;
      for (int i = lane; i < count; i += 32) c += ((uint32_t)(ent[i] >> 32) >= candT) ? 1 : 0;
      c = __reduce_add_sync(0xffffffffu, c);
      if (c >= p.k) T = candT;
    }
    const uint32_t band_key = f2ord(ord2f(T) - e2);
    if (band_key > g_key) g_key = band_key;
    int kept = 0;
    for (int base = 0; base < count; base += 32) {
      const int i = base + lane;
      unsigned long long e = 0;
      bool keep = false;
      if (i < count) { e = ent[i]; keep = (uint32_t)(e >> 32) > g_key; }
      const unsigned bal = __ballot_sync(0xffffffffu, keep);
      __syncwarp();
      if (keep) ent[kept + __popc(bal & ((1u << lane) - 1u))] = e;
      kept += __popc(bal);
      __syncwarp();
    }
    return kept;
  };
  // All stream counts in one load (lane s holds stream s; SS <= 32); the streams' entries are
  // then read as ONE flattened list, four independent 32-entry loads in flight per step -- a
  // serial count -> entries -> count chain per stream cost 13 % of the kernel in load latency.
  const int my_c = (lane < p.SS) ? p.cand_cnt[(size_t)q * p.SS + lane] : 0;
  if (__any_sync(0xffffffffu, my_c < 0)) bad = true;
  int incl = my_c;                                   // inclusive prefix sum of the counts
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  const int total = bad ? 0 : __shfl_sync(0xffffffffu, incl, 31);
  const uint2* qsrc = p.cand + (size_t)q * p.SS * p.cap;
  auto fetch = [&](int j, uint32_t& key, uint32_t& idx) -> bool {     // flattened entry j
    // stream = number of inclusive prefixes <= j (all lanes take part in the shuffles)
    int st = 0, before = 0;
    for (int t = 0; t < p.SS; ++t) {
      const int pre = __shfl_sync(0xffffffffu, incl, t);
      if (pre <= j) { ++st; before = pre; }
    }
    if (j >= total) return false;
    const uint2 e = qsrc[(size_t)st * p.cap + (j - before)];
    key = f2ord(__uint_as_float(e.x));
    idx = e.y;
    return true;
  };
  for (int base = 0; base < total && !bad; base += 128) {
    uint32_t key[4], idx[4];
    bool ok[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) { key[u] = 0; idx[u] = 0; ok[u] = false; }
    // (shuffles inside fetch need all lanes: every lane calls it, out-of-range ones get false)
#pragma unroll
    for (int u = 0; u < 4; ++u) ok[u] = fetch(base + 32 * u + lane, key[u], idx[u]);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (base + 32 * u >= total) break;               // uniform
      if (M + 32 > per_warp_entries) {
        __syncwarp();
        M = tighten(M);
        if (M + 32 > per_warp_entries) { bad = true; break; }
      }
      const bool keep = ok[u] && key[u] > g_key;
      const unsigned bal = __ballot_sync(0xffffffffu, keep);
      if (keep) ent[M + __popc(bal & ((1u << lane) - 1u))] = ((unsigned long long)key[u] << 32) | idx[u];
      M += __popc(bal);
    }
  }
  __syncwarp();
  // fewer than k survivors: impossible for finite inputs with this shard's own thresholds (the
  // exact path decides), legitimate under a cross-shard bound (the rest of the list is padding)
  if (M < p.k && !p.allow_partial) bad = true;
  int n_s = 0;
  if (!bad) {
    n_s = (M < p.k) ? M : tighten(M);       // (the band needs k entries to be defined)
    if (n_s > RR_MAX) bad = true;
  }
  if (bad) {
    if (lane == 0) p.fb_list[atomicAdd(&p.counters[0], 1)] = (int)q;
    return;
  }
  // ---- exact cosine of every survivor
  double qh[VPL];
  const double nq = p.q_nrm[q];
  const float* qp = p.query + q * p.ldq;
#pragma unroll
  for (int t = 0; t < VPL; ++t) {
    const int d = VEC ? (4 * lane + 128 * (t >> 2) + (t & 3)) : (lane + 32 * t);
    qh[t] = d < p.dim ? (double)__ldg(qp + d) : 0.0;
  }
  // RPI independent row gathers in flight per warp: the phase is DRAM-latency bound otherwise
  const double ss_q = nq * nq;
  for (int i = 0; i < n_s; i += RPI) {
    uint32_t r[RPI];
    double acc[RPI];
    float l1[RPI];
#pragma unroll
    for (int u = 0; u < RPI; ++u) r[u] = (uint32_t)ent[min(i + u, n_s - 1)];
#pragma unroll
    for (int u = 0; u < RPI; ++u)
      acc[u] = row_dot<VEC, WANT_L1, VPL>(p.bank + (int64_t)r[u] * p.ldb, qh, p.dim, lane, &l1[u]);
#pragma unroll
    for (int u = 0; u < RPI; ++u) acc[u] = warp_sum(acc[u]);
    if (want_l1) {
#pragma unroll
      for (int u = 0; u < RPI; ++u) l1[u] = warp_sum(l1[u]);
    }
    __syncwarp();
    double a = acc[0];
    uint32_t rr = r[0];
    float l1v = want_l1 ? l1[0] : 0.f;
#pragma unroll
    for (int u = 1; u < RPI; ++u)
      if (lane == u) { a = acc[u]; rr = r[u]; if (want_l1) l1v = l1[u]; }
    if (lane < RPI && i + lane < n_s) {
      const double ns = p.bank_nrm[rr];
      const float v = (float)(a / (nq * ns));
      ent[i + lane] = ((unsigned long long)f2ord(v) << 32) | (unsigned long long)(0xffffffffu - rr);
      if (want_dist) {
        float d = l1v;
        if (!want_l1) {               // ||s - q||^2 = |s|^2 + |q|^2 - 2 s.q, all in fp64
          const double ss = ns * ns + ss_q;
          const double d2 = ss - 2.0 * a;
          d = d2 <= 1e-12 * ss ? 0.f : (float)sqrt(d2);
        }
        pay[i + lane] = d;
      }
    }
    __syncwarp();
  }
  __syncwarp();
  // ---- sort (value desc, index asc)
  int P = 1;
  while (P < n_s) P <<= 1;
  for (int j = n_s + lane; j < P; j += 32) ent[j] = 0ull;
  if (want_dist)
    for (int j = lane; j < P; j += 32) slot[j] = (unsigned short)j;
  __syncwarp();
  for (int size = 2; size <= P; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = lane; t < (P >> 1); t += 32) {
        const int lo = 2 * t - (t & (stride - 1));
        const int hi = lo + stride;
        const bool desc = ((lo & size) == 0);
        const unsigned long long a = ent[lo], b = ent[hi];
        if ((a < b) == desc) {
          ent[lo] = b; ent[hi] = a;
          if (want_dist) { const unsigned short t2 = slot[lo]; slot[lo] = slot[hi]; slot[hi] = t2; }
        }
      }
      __syncwarp();
    }
  }
  // speculative start (spec_rank): every row it dropped scores at most spec + eps exactly, so the
  // result stands iff the k-th best found lies strictly above that; otherwise the exact path decides
  {
    const float sp = p.spec ? p.spec[q] : -INFINITY;
    if (sp > -INFINITY) {
      const float vk = (n_s >= p.k) ? ord2f((uint32_t)(ent[p.k - 1] >> 32)) : -INFINITY;
      if (!(vk > sp + 0.5f * e2)) {
        if (lane == 0) { p.fb_list[atomicAdd(&p.counters[0], 1)] = (int)q; atomicAdd(&p.counters[2], 1); }
        return;
      }
    }
  }
  for (int j = lane; j < p.k; j += 32) {
    if (j < n_s) {
      const unsigned long long e = ent[j];
      p.out_idx[q * p.k + j] = (int64_t)(0xffffffffu - (uint32_t)e) + p.index_offset;
      if (p.out_val) p.out_val[q * p.k + j] = ord2f((uint32_t)(e >> 32));
      if (want_dist) p.out_dist[q * p.k + j] = pay[slot[j]];
    } else {                       // padding of a partial list: loses every merge
      p.out_idx[q * p.k + j] = 0x7fffffffll;
      if (p.out_val) p.out_val[q * p.k + j] = -INFINITY;
      if (want_dist) p.out_dist[q * p.k + j] = INFINITY;
    }
  }
  if (lane == 0) atomicAdd(&p.counters[1], 1);
}

// ============================================================================ host side
int tc_cap_for_k(int k) { return k <= 192 ? 256 : (k <= 896 ? 1024 : 0); }

void tc_workspace(Arena& a, int64_t n_bank, int64_t n_query, int dim, int top_k, TcWorkspace& w) {
  const int nkb = (dim + 63) / 64;
  w.nkb = nkb;
  w.e_acc = nkb <= 4 ? E_ACC : E_ACC_WIDE;
  w.q_pad = (int64_t)align_up((size_t)n_query, 128);
  w.n_pad = (int64_t)align_up((size_t)n_bank, ST_BN);
  w.plan = plan_lanes(w.q_pad / 128, w.n_pad / ST_BN, sm_count(), ST_MAX_SLOTS);
  w.SS = w.plan.slots * ST_CP;
  w.cap = tc_cap_for_k(top_k);
  // everything derived from the bank first: its offsets do not depend on the query count, so a
  // resident bank (MCLST_FM_BANK_PACKED) stays valid across calls with different query batches
  w.stats = a.take<uint32_t>(16);
  w.bpack = a.take<uint8_t>(tilepack_bytes(w.n_pad, nkb * 64));
  w.b_nrm = a.take<double>((size_t)w.n_pad);
  w.b_resid = a.take<float>((size_t)w.n_pad);
  w.qpack = a.take<uint8_t>(tilepack_bytes(w.q_pad, nkb * 64));
  w.q_nrm = a.take<double>((size_t)w.q_pad);
  w.q_resid = a.take<float>((size_t)w.q_pad);
  w.gthr = a.take<uint32_t>((size_t)w.q_pad);
  w.spec = a.take<float>((size_t)w.q_pad);
  w.speculate = 1;
  w.cand = a.take<uint2>((size_t)w.q_pad * w.SS * w.cap);
  w.cand_cnt = a.take<int>((size_t)w.q_pad * w.SS);
  w.fb_list = a.take<int>((size_t)n_query);
  // seed pass: a strided sample of the bank tiles -- 1/8 of them, at most 128 (3.3 % of the main
  // pass at 1M rows, 6.5 % for a 500k-row shard).  A thinner sample was tried for shards (1/24):
  // seed pass 1.41 -> 1.04 ms but main pass 13.5 -> 14.7 ms at 500k rows -- the looser start costs
  // more than the sample saves.
  const int64_t tiles = w.n_pad / ST_BN;
  int n_seed = (int)std::min<int64_t>(128, tiles / 8);
  if (n_seed * 8 < 2 * top_k) n_seed = 0;
  w.n_seed = n_seed;
  w.seed = n_seed ? a.take<float>((size_t)w.q_pad * n_seed * 8) : nullptr;
}

int launch_pack_rows(const float* x, int64_t rows, int64_t rows_pad, int64_t ld, int dim, int nkb,
                     uint8_t* packed, double* nrm, float* resid, uint32_t* stats, cudaStream_t st) {
  const int wpb = 8;
  const bool vec = (dim % 8 == 0) && (ld % 4 == 0) && ((uintptr_t)x % 16 == 0);
  const unsigned grid = (unsigned)std::min<int64_t>(ceil_div(rows_pad, wpb), (int64_t)sm_count() * 8 * 4);
  MCLST_REQUIRE(nkb >= 1 && nkb * 64 <= TC_MAX_DIM, MCLST_ERR_UNSUPPORTED, "pack_rows: %d K blocks", nkb);
  auto kern = nkb <= 4 ? (vec ? pack_rows_kernel<true, 1> : pack_rows_kernel<false, 1>)
                       : (vec ? pack_rows_kernel<true, 2> : pack_rows_kernel<false, 2>);
  kern<<<grid, wpb * 32, 0, st>>>(x, rows, rows_pad, ld, dim, nkb, packed, nrm, resid, stats);
  MCLST_LAUNCH_CHECK();
  return 0;
}

template <int CAP, SimPass PASS>
static int launch_lanes(const SimParams& p, const LanePlan& L, cudaStream_t st) {
  const bool wide = p.nkb > ST_A_BYTES / TP_SLICE_BYTES;
  auto kern = wide ? sim_topk_lanes_kernel<CAP, PASS, ST_A_BYTES_WIDE, ST_STAGES_WIDE>
                   : sim_topk_lanes_kernel<CAP, PASS, ST_A_BYTES, ST_STAGES>;
  const int smem = wide ? st_smem(ST_A_BYTES_WIDE, ST_STAGES_WIDE) : st_smem(ST_A_BYTES, ST_STAGES);
  MCLST_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  kern<<<(unsigned)L.W, ST_THREADS, smem, st>>>(p, L);
  MCLST_LAUNCH_CHECK();
  return 0;
}

static SimParams sim_params(const TcWorkspace& w, int64_t n_bank, int64_t n_query, int top_k) {
  SimParams p{};
  p.qpack = w.qpack; p.bpack = w.bpack; p.nkb = w.nkb; p.Q = n_query; p.N = n_bank;
  p.tiles_total = (int)(w.n_pad / ST_BN); p.k = top_k; p.e_acc = w.e_acc;
  p.q_resid = w.q_resid; p.bank_stats = w.stats; p.cand = w.cand; p.cand_cnt = w.cand_cnt;
  p.gthr = w.gthr;
  return p;
}

// Speculative warm start.  The guaranteed seed threshold is the k-th largest value of the sample
// (k sampled rows score at least that): global rank ~ k / f for a sampled fraction f, i.e. ~1500
// at cfg4, where 97 % of the 32-score chunks still hold a passing element.  Starting from the
// j-th largest instead (rank ~ j / f) is valid exactly when fewer than j of the true top k-1 rows
// fell into the sample -- X ~ Binomial(k-1, f) for a bank in no particular order.  j is the
// smallest rank with P(X >= j) < 1e-7 per query; the re-rank checks the outcome (the k-th best
// exact score found must lie above threshold + eps, else nothing dropped could have mattered is
// NOT guaranteed and the query is recomputed by the exact path), so a bank whose order defeats the
// binomial model costs time, never correctness.
int spec_rank(int k, double f) {
  if (!(f > 0.0) || f >= 0.5 || k < 8) return k;
  const int n = k - 1;
  // P(X >= j) summed from the top, every term from its logarithm (f^n underflows a double long
  // before the terms that matter: k = 200, f = 0.03)
  const double lf = log(f), l1f = log1p(-f), lgn = lgamma((double)n + 1.0);
  double tail = 0.0;
  int best = k;
  for (int j = n; j >= 1; --j) {
    tail += exp(lgn - lgamma((double)j + 1.0) - lgamma((double)(n - j) + 1.0) + j * lf + (n - j) * l1f);
    if (tail < 1e-7) best = j;
    else break;
  }
  return std::max(4, std::min(best, k));
}

int launch_sim_topk(const TcWorkspace& w, int64_t n_bank, int64_t n_query, int top_k, cudaStream_t st,
                    int phase, const SeedBounds* sb) {
  // phase 0: seed pass + main pass; 1: thresholds reset + seed pass only (optionally writing the
  // cross-shard bounds of sb); 2: main pass only, after applying sb->ext_bound when given
  const SimParams p = sim_params(w, n_bank, n_query, top_k);
  if (phase != 2) MCLST_CUDA(cudaMemsetAsync(w.gthr, 0, (size_t)w.q_pad * sizeof(uint32_t), st));
  const bool seeded = w.n_seed > 0;
  if (phase == 1 && !seeded && sb) {       // no sample: no bound to offer
    if (sb->bound_k) fill_kernel<<<(unsigned)ceil_div(n_query, 256), 256, 0, st>>>(sb->bound_k, n_query, -INFINITY);
    if (sb->bound_part) fill_kernel<<<(unsigned)ceil_div(n_query, 256), 256, 0, st>>>(sb->bound_part, n_query, -INFINITY);
    MCLST_LAUNCH_CHECK();
  }
  if (phase == 2 && sb && sb->ext_bound) {
    apply_bound_kernel<<<(unsigned)ceil_div(n_query, 256), 256, 0, st>>>(sb->ext_bound, n_query, w.q_resid,
                                                                        w.stats, w.gthr, w.e_acc);
    MCLST_LAUNCH_CHECK();
  }
  if (seeded && phase != 2) {
    // ---- seed pass, on balanced unit lists of its own over the sampled tiles
    SimParams sp = p;
    sp.seed_out = w.seed; sp.n_tiles = w.n_seed; sp.tile_begin = 0;
    sp.tile_stride = std::max(1, p.tiles_total / w.n_seed);
    int rc = launch_lanes<256, SimPass::Seed>(sp, plan_lanes(w.q_pad / 128, w.n_seed, sm_count(), 4), st);
    if (rc) return rc;
    // bounds that other shards will rely on must be guaranteed ones: no speculation when staged
    const bool speculate = w.speculate && !(sb && (sb->bound_k || sb->bound_part));
    const int k_seed = speculate ? spec_rank(top_k, (double)w.n_seed / (double)p.tiles_total) : top_k;
    seed_threshold_kernel<<<(unsigned)ceil_div(n_query, 4), 128, 0, st>>>(
        w.seed, w.n_seed * 8, n_query, k_seed, w.q_resid, w.stats, w.gthr, sb ? std::max(1, sb->k_part) : 1,
        sb ? sb->bound_k : nullptr, sb ? sb->bound_part : nullptr, k_seed < top_k ? w.spec : nullptr, w.e_acc);
    MCLST_LAUNCH_CHECK();
    if (k_seed >= top_k) MCLST_CUDA(cudaMemsetAsync(w.spec, 0xff, (size_t)w.q_pad * sizeof(float), st));  // NaN: none
  } else if (phase != 2) {
    MCLST_CUDA(cudaMemsetAsync(w.spec, 0xff, (size_t)w.q_pad * sizeof(float), st));
  }
  if (phase == 1) return 0;
  // slots a query block does not use must read as empty
  MCLST_CUDA(cudaMemsetAsync(w.cand_cnt, 0, (size_t)w.q_pad * w.SS * sizeof(int), st));
  if (w.cap == 256) return launch_lanes<256, SimPass::Candidates>(p, w.plan, st);
  // large-k configurations (reference k = 200 / 600) are small problems: one variant
  if (w.cap == 1024) return launch_lanes<1024, SimPass::Candidates>(p, w.plan, st);
  MCLST_REQUIRE(false, MCLST_ERR_UNSUPPORTED, "sim_topk: cap %d", w.cap);
}

int launch_sim_dump(const TcWorkspace& w, int64_t n_bank, int64_t n_query, float* dump, int64_t dump_ld,
                    cudaStream_t st) {
  SimParams p = sim_params(w, n_bank, n_query, 1);
  p.dump = dump; p.dump_ld = dump_ld;
  // the epilogue reads the shared thresholds whatever the pass: keep them defined
  MCLST_CUDA(cudaMemsetAsync(w.gthr, 0, (size_t)w.q_pad * sizeof(uint32_t), st));
  return launch_lanes<256, SimPass::Dump>(p, w.plan, st);
}

int launch_apply_bound(const TcWorkspace& w, int64_t n_query, const float* ext_bound, cudaStream_t st) {
  apply_bound_kernel<<<(unsigned)ceil_div(n_query, 256), 256, 0, st>>>(ext_bound, n_query, w.q_resid, w.stats, w.gthr,
                                                                      w.e_acc);
  MCLST_LAUNCH_CHECK();
  return 0;
}
int launch_export_bound(const TcWorkspace& w, int64_t n_query, int top_k, float* bound, int k_part,
                        float* bound_part, cudaStream_t st) {
  export_bound_kernel<<<(unsigned)ceil_div(n_query, 4), 128, 0, st>>>(w.cand, w.cand_cnt, w.SS, w.cap, top_k, w.gthr,
                                                                     n_query, w.q_resid, w.stats, bound,
                                                                     std::max(1, std::min(k_part, top_k)), bound_part,
                                                                     w.e_acc);
  MCLST_LAUNCH_CHECK();
  return 0;
}

int launch_rerank(const TcWorkspace& w, const float* bank, int64_t n_bank, int64_t ldb,
                  const float* query, int64_t n_query, int64_t ldq, int dim, int top_k,
                  int64_t index_offset, int64_t* out_idx, float* out_val, float* out_dist, int dist_p,
                  int* counters, cudaStream_t st, bool allow_partial) {
  RerankParams p;
  p.allow_partial = allow_partial ? 1 : 0;
  p.spec = allow_partial ? nullptr : w.spec;
  p.cand = w.cand; p.cand_cnt = w.cand_cnt; p.SS = w.SS; p.cap = w.cap; p.k = top_k; p.e_acc = w.e_acc;
  p.Q = n_query; p.N = n_bank; p.bank = bank; p.ldb = ldb; p.bank_nrm = w.b_nrm;
  p.query = query; p.ldq = ldq; p.q_nrm = w.q_nrm; p.q_resid = w.q_resid;
  p.bank_stats = w.stats; p.q_stats = w.stats + 8; p.gthr = w.gthr; p.dim = dim;
  p.index_offset = index_offset;
  p.out_idx = out_idx; p.out_val = out_val; p.out_dist = out_dist; p.dist_p = dist_p;
  p.fb_list = w.fb_list; p.counters = counters;
  // shared memory: per warp a power-of-two number of 8-byte entries (bitonic sort), at most 4096;
  // a query whose streams hold more than that goes to the exact path
  int per_warp = 1;
  while (per_warp < w.SS * w.cap && per_warp < 1024) per_warp <<= 1;
  if (per_warp < 2 * top_k) per_warp = 2048;
  int wpb = 4;
  while (wpb > 1 && (size_t)wpb * per_warp * 8 > 64 * 1024) wpb >>= 1;
  const size_t smem = (size_t)wpb * per_warp * 8 + (size_t)wpb * RR_MAX * 6;
  const bool wide = dim > 256;
  const bool vec = (dim == (wide ? 512 : 256)) && (ldb % 4 == 0) && (ldq % 4 == 0) && ((uintptr_t)bank % 16 == 0) &&
                   ((uintptr_t)query % 16 == 0);
  const bool l1 = out_dist != nullptr && dist_p == 1;
  const unsigned grid = (unsigned)ceil_div(n_query, wpb);
  auto launch = [&](auto kern, size_t& attr) -> int {
    if (smem > attr) {
      MCLST_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)std::max<size_t>(smem, 48 * 1024)));
      attr = smem;
    }
    kern<<<grid, 128, smem, st>>>(p, wpb, per_warp);
    return 0;
  };
  static size_t attr[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  int rc;
  if (wide) {
    if (vec) rc = l1 ? launch(rerank_kernel<true, true, 16>, attr[7]) : launch(rerank_kernel<true, false, 16>, attr[6]);
    else rc = l1 ? launch(rerank_kernel<false, true, 16>, attr[5]) : launch(rerank_kernel<false, false, 16>, attr[4]);
  } else {
    if (vec) rc = l1 ? launch(rerank_kernel<true, true, 8>, attr[3]) : launch(rerank_kernel<true, false, 8>, attr[2]);
    else rc = l1 ? launch(rerank_kernel<false, true, 8>, attr[1]) : launch(rerank_kernel<false, false, 8>, attr[0]);
  }
  if (rc) return rc;
  MCLST_LAUNCH_CHECK();
  return 0;
}

}  // namespace mclst

extern "C" int mclst_debug_spec_rank(int top_k, double sampled_fraction) {
  return mclst::spec_rank(top_k, sampled_fraction);
}

extern "C" int mclst_debug_lane_plan(int64_t query_blocks, int64_t bank_tiles, int lanes, int max_slots,
                                     int* units, int64_t max_units, int64_t* n_units, int* slots) {
  using namespace mclst;
  MCLST_REQUIRE(query_blocks >= 1 && bank_tiles >= 1 && lanes >= 1 && max_slots >= 1 && n_units && slots,
                MCLST_ERR_INVALID, "debug_lane_plan: bad args");
  const LanePlan L = plan_lanes(query_blocks, bank_tiles, lanes, max_slots);
  *slots = L.slots;
  int64_t n = 0;
  for (int c = 0; c < L.W; ++c) {
    LaneUnit u;
    for (int j = 0; lane_unit(L, (int)bank_tiles, c, j, u); ++j, ++n) {
      if (units && n < max_units) {
        int* o = units + 5 * n;
        o[0] = c; o[1] = u.qb; o[2] = u.t0; o[3] = u.t1; o[4] = u.slot;
      }
    }
  }
  *n_units = n;
  return 0;
}
