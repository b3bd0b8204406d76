// Internal declarations shared by the retrieval translation units.
#pragma once
#include "common.cuh"

namespace mclst {

int launch_row_norms(const float* x, int64_t rows, int64_t ld, int dim, double* nrm, cudaStream_t st);

int exact_topk_ctas(int64_t n_bank, int64_t n_query);
size_t exact_topk_scratch_floats(int64_t n_bank, int64_t n_query);
// qlist/qcount_ptr (device) select a subset of queries; when both are null queries
// 0..qcount-1 are processed.  n_query_cap bounds the subset size (grid / scratch sizing).
int launch_exact_topk(const float* bank, int64_t N, int64_t ldb, const double* bank_nrm,
                      const float* query, int64_t ldq, const double* q_nrm, int dim,
                      const int* qlist, const int* qcount_ptr, int qcount, int64_t n_query_cap,
                      int k, int64_t index_offset, float* scratch, int64_t* out_idx,
                      float* out_val, cudaStream_t st);

// ---- tensor-core candidate path (sim_topk.cu)
constexpr int TC_MAX_DIM = 512;   // widest rows it takes (the resident query block of the wide variant)
// Work decomposition of the persistent candidate kernel: W lanes (CTAs) walk closed-form unit
// lists (sim_topk.cu: plan_lanes / lane_unit); `slots` candidate slots per query block.
struct LanePlan {
  int W, rounds, rest, w, R, M, Lt, slots;
  int h, hm;      // sub-units (= fresh candidate buffers) per full-round unit / per main-lane unit
};
struct TcWorkspace {
  int nkb, SS, cap;         // SS = 2 * plan.slots candidate streams per query (two column halves)
  float e_acc;              // accumulation bound of this width (sim_topk.cu: E_ACC, E_ACC_WIDE)
  LanePlan plan;            // of the candidate pass
  int64_t q_pad, n_pad;
  uint32_t* stats;          // [0..7] bank: max residual bits, non-finite flag; [8..15] queries
  uint8_t *qpack, *bpack;
  double *q_nrm, *b_nrm;
  float *q_resid, *b_resid;
  uint32_t* gthr;
  float* spec;      // [q_pad] speculative start threshold of the seed pass (NaN: none), checked by the re-rank
  int speculate;    // 0: guaranteed thresholds only (MCLST_FM_NO_SPECULATION)
  uint2* cand;
  int* cand_cnt;
  int* fb_list;
  float* seed;      // chunk maxima of the seed pass [q_pad][n_seed * 8]
  int n_seed;
};
int tc_cap_for_k(int k);
void tc_workspace(Arena& a, int64_t n_bank, int64_t n_query, int dim, int top_k, TcWorkspace& w);
int launch_pack_rows(const float* x, int64_t rows, int64_t rows_pad, int64_t ld, int dim, int nkb,
                     uint8_t* packed, double* nrm, float* resid, uint32_t* stats, cudaStream_t st);
// cross-shard exchange around the seed pass (sim_topk.cu): outputs of phase 1, input of phase 2
struct SeedBounds {
  int k_part;              // bound_part is about the k_part-th best of this shard's sample
  float* bound_k;          // [Q] >= k rows of this shard have an exact score >= bound_k[q] (-inf: unknown)
  float* bound_part;       // [Q] same for k_part rows
  const float* ext_bound;  // [Q] lower bound of the exact GLOBAL k-th best score, or null
};
int launch_sim_topk(const TcWorkspace& w, int64_t n_bank, int64_t n_query, int top_k, cudaStream_t st,
                    int phase = 0, const SeedBounds* sb = nullptr);
// testing aid: the raw tensor-core similarities of the packed operands into dump [n_query, dump_ld]
int launch_sim_dump(const TcWorkspace& w, int64_t n_bank, int64_t n_query, float* dump, int64_t dump_ld,
                    cudaStream_t st);
int launch_apply_bound(const TcWorkspace& w, int64_t n_query, const float* ext_bound, cudaStream_t st);
int launch_export_bound(const TcWorkspace& w, int64_t n_query, int top_k, float* bound, int k_part,
                        float* bound_part, cudaStream_t st);
int launch_rerank(const TcWorkspace& w, const float* bank, int64_t n_bank, int64_t ldb,
                  const float* query, int64_t n_query, int64_t ldq, int dim, int top_k,
                  int64_t index_offset, int64_t* out_idx, float* out_val, float* out_dist, int dist_p,
                  int* counters, cudaStream_t st, bool allow_partial = false);
// distances of the winners of the queries in qlist (exact-fallback rows) or of all queries
int launch_neighbor_distances(const float* spot_key, int64_t n_bank, int64_t ld_key, const float* query,
                              int64_t n_query, int64_t ld_query, int dim, const int64_t* indices, int k,
                              int64_t index_offset, int p, float* out_dist, const int* qlist,
                              const int* qcount_ptr, cudaStream_t st);

}  // namespace mclst
