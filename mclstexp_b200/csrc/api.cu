// extern "C" surface of libmclst_b200.so: error plumbing + retrieval orchestration.
#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <vector>
#include "common.cuh"
#include "retrieval.cuh"

namespace mclst {

static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// ---- per-kernel event trace ------------------------------------------------------------
struct ProfMark { cudaEvent_t ev; const char* name; cudaStream_t st; };
static bool g_prof_on = false;
static std::vector<ProfMark> g_marks;
static std::vector<cudaEvent_t> g_pool;
static std::mutex g_prof_mu;

void prof_mark(cudaStream_t st, const char* name) {
  if (!g_prof_on) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  cudaEvent_t ev;
  if (!g_pool.empty()) { ev = g_pool.back(); g_pool.pop_back(); }
  else if (cudaEventCreate(&ev) != cudaSuccess) return;
  cudaEventRecord(ev, st);
  g_marks.push_back({ev, name, st});
}

int sm_count() {
  static int cached = 0;
  if (!cached) {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
      cached = n;
    else
      return 148;
  }
  return cached;
}

// Layout of the find_matches workspace.  The first 256 bytes are int32 counters:
// [0] queries recomputed by the exact brute-force path, [1] queries resolved by the
// tensor-core path.
struct FmWorkspace {
  int* counters;
  bool use_tc;
  TcWorkspace tc;
  double* bank_nrm;
  double* q_nrm;
  float* scratch;
  size_t bytes;
};

// The one eligibility rule of the tensor-core candidate path (exported as
// mclst_find_matches_tc_eligible; the Python layers ask it instead of restating it).
static bool tc_eligible(int64_t n_bank, int dim, int top_k, int flags) {
  return !(flags & MCLST_FM_EXACT_ONLY) && dim >= 1 && dim <= TC_MAX_DIM && tc_cap_for_k(top_k) != 0 &&
         n_bank >= top_k;
}

static FmWorkspace carve_fm(void* ws, size_t cap, int64_t n_bank, int64_t n_query, int dim,
                            int top_k, int flags) {
  Arena a(ws, cap);
  FmWorkspace w{};
  w.counters = a.take<int>(64);
  w.use_tc = tc_eligible(n_bank, dim, top_k, flags);
  if (w.use_tc) {
    tc_workspace(a, n_bank, n_query, dim, top_k, w.tc);
    w.tc.speculate = (flags & MCLST_FM_NO_SPECULATION) ? 0 : 1;
    w.bank_nrm = w.tc.b_nrm;
    w.q_nrm = w.tc.q_nrm;
  } else {
    w.bank_nrm = a.take<double>((size_t)n_bank);
    w.q_nrm = a.take<double>((size_t)n_query);
  }
  w.scratch = a.take<float>(exact_topk_scratch_floats(n_bank, n_query));
  w.bytes = align_up(a.off, 256);
  return w;
}

}  // namespace mclst

using namespace mclst;

extern "C" int mclst_version(void) { return 100; }
extern "C" const char* mclst_last_error(void) { return g_err; }
extern "C" int64_t mclst_launch_count(void) { return g_launches.load(); }

extern "C" int mclst_device_info(int* sms, int* major, int* minor) {
  int dev = 0;
  MCLST_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp p;
  MCLST_CUDA(cudaGetDeviceProperties(&p, dev));
  if (sms) *sms = p.multiProcessorCount;
  if (major) *major = p.major;
  if (minor) *minor = p.minor;
  MCLST_REQUIRE(p.major == 10, MCLST_ERR_DEVICE, "device is sm_%d%d, this library is sm_100a only",
                p.major, p.minor);
  return 0;
}

extern "C" int mclst_profile_enable(int on) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof_on = on != 0;
  for (auto& m : g_marks) g_pool.push_back(m.ev);
  g_marks.clear();
  return 0;
}

// Synchronises the device, then writes up to `cap` records: names_out[i] (<= 47 chars + NUL,
// 48-byte stride) and ms_out[i] = time from mark i to mark i+1 (the last mark of a call is
// named "end" and closes the previous kernel).  Returns the number of records via *n.
extern "C" int mclst_profile_collect(char* names_out, float* ms_out, int cap, int* n) {
  MCLST_REQUIRE(names_out && ms_out && n, MCLST_ERR_INVALID, "profile_collect: null pointer");
  MCLST_CUDA(cudaDeviceSynchronize());
  std::lock_guard<std::mutex> lk(g_prof_mu);
  int cnt = 0;
  for (size_t i = 0; i + 1 < g_marks.size() && cnt < cap; ++i) {
    if (!strcmp(g_marks[i].name, "end")) continue;
    // the next mark on the SAME stream closes this one (calls may interleave two streams)
    size_t j = i + 1;
    while (j < g_marks.size() && g_marks[j].st != g_marks[i].st) ++j;
    if (j == g_marks.size()) continue;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, g_marks[i].ev, g_marks[j].ev) != cudaSuccess) continue;
    strncpy(names_out + 48 * cnt, g_marks[i].name, 47);
    names_out[48 * cnt + 47] = 0;
    ms_out[cnt++] = ms;
  }
  for (auto& m : g_marks) g_pool.push_back(m.ev);
  g_marks.clear();
  *n = cnt;
  return 0;
}

extern "C" int mclst_read_counters(const void* workspace, int64_t out[4], mclst_stream_t stream) {
  MCLST_REQUIRE(workspace && out, MCLST_ERR_INVALID, "read_counters: null pointer");
  int c[4] = {0, 0, 0, 0};
  MCLST_CUDA(cudaMemcpyAsync(c, workspace, sizeof(c), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  MCLST_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  out[0] = c[1];   // tensor-core path
  out[1] = c[0];   // exact fallback
  out[2] = c[2];   // of the fallbacks: speculative seeds that did not verify
  out[3] = c[3];
  return 0;
}

extern "C" int mclst_find_matches_workspace_bytes(int64_t n_bank, int64_t n_query, int dim,
                                                  int top_k, int flags, size_t* bytes) {
  MCLST_REQUIRE(bytes, MCLST_ERR_INVALID, "workspace_bytes: null pointer");
  MCLST_REQUIRE(n_bank >= 0 && n_query >= 0 && dim >= 1 && top_k >= 1, MCLST_ERR_INVALID,
                "workspace_bytes: bad shape");
  *bytes = carve_fm(nullptr, 0, n_bank, n_query, dim, top_k, flags).bytes;
  return 0;
}

extern "C" int mclst_find_matches_tc_eligible(int64_t n_bank, int dim, int top_k, int flags) {
  return tc_eligible(n_bank, dim, top_k, flags) ? 1 : 0;
}

extern "C" int mclst_find_matches_dist(const float* bank, int64_t n_bank, int64_t ld_bank,
                                       const float* query, int64_t n_query, int64_t ld_query,
                                       int dim, int top_k, int64_t index_offset,
                                       int64_t* out_indices, float* out_values,
                                       float* out_distances, int dist_p, void* workspace,
                                       size_t workspace_bytes, int flags, mclst_stream_t stream);

extern "C" int mclst_find_matches(const float* bank, int64_t n_bank, int64_t ld_bank,
                                  const float* query, int64_t n_query, int64_t ld_query, int dim,
                                  int top_k, int64_t index_offset, int64_t* out_indices,
                                  float* out_values, void* workspace, size_t workspace_bytes,
                                  int flags, mclst_stream_t stream) {
  return mclst_find_matches_dist(bank, n_bank, ld_bank, query, n_query, ld_query, dim, top_k,
                                 index_offset, out_indices, out_values, nullptr, 2, workspace,
                                 workspace_bytes, flags, stream);
}

// The stages of find_matches.  stage bits: 1 = pack (+ thresholds reset + seed pass, writing the
// cross-shard bounds when asked), 2 = candidate (main tensor-core) pass, 4 = re-rank + exact
// fallback.  The single-call entry runs all of them; bank shards run them separately with a bound
// exchange in between (sb->ext_bound is applied at the start of the first stage of a call that is
// not stage 1; bound_k receives the post-candidate bound when a call ends with stage 2).
static int find_matches_stages(int stages, const float* bank, int64_t n_bank, int64_t ld_bank,
                               const float* query, int64_t n_query, int64_t ld_query, int dim,
                               int top_k, int64_t index_offset, int64_t* out_indices,
                               float* out_values, float* out_distances, int dist_p,
                               SeedBounds* sb, void* workspace, size_t workspace_bytes, int flags,
                               cudaStream_t st) {
  MCLST_REQUIRE(dist_p == 1 || dist_p == 2, MCLST_ERR_INVALID, "find_matches: dist_p must be 1 or 2");
  MCLST_REQUIRE(bank && workspace && (query || n_query == 0), MCLST_ERR_INVALID, "find_matches: null pointer");
  MCLST_REQUIRE(!(stages & 4) || out_indices || n_query == 0, MCLST_ERR_INVALID, "find_matches: null output");
  MCLST_REQUIRE(dim >= 1 && ld_bank >= dim && (ld_query >= dim || n_query == 0), MCLST_ERR_INVALID,
                "find_matches: bad dim/ld");
  // torch.topk raises when k exceeds the dimension (evel_her2st.py:82)
  MCLST_REQUIRE(top_k >= 1 && top_k <= n_bank, MCLST_ERR_INVALID,
                "find_matches: top_k %d out of range for %lld bank rows", top_k, (long long)n_bank);
  MCLST_REQUIRE(n_bank < (1ll << 31), MCLST_ERR_UNSUPPORTED, "find_matches: bank shard too large");
  FmWorkspace w = carve_fm(workspace, workspace_bytes, n_bank, n_query, dim, top_k, flags);
  MCLST_REQUIRE(w.bytes <= workspace_bytes, MCLST_ERR_WORKSPACE,
                "find_matches: workspace %zu < %zu", workspace_bytes, w.bytes);
  const bool packed = (flags & MCLST_FM_BANK_PACKED) != 0;
  MCLST_REQUIRE(!packed || w.use_tc, MCLST_ERR_INVALID,
                "find_matches: MCLST_FM_BANK_PACKED needs the tensor-core path (dim <= %d, k <= 896, k <= n_bank)",
                TC_MAX_DIM);
  int rc;
  if (!w.use_tc) {
    if (stages & 1) {
      if (sb && sb->bound_k) MCLST_CUDA(cudaMemsetAsync(sb->bound_k, 0xff, (size_t)n_query * 4, st));     // -NaN: "unknown"
      if (sb && sb->bound_part) MCLST_CUDA(cudaMemsetAsync(sb->bound_part, 0xff, (size_t)n_query * 4, st));
    }
    if ((stages & 2) && !(stages & 4) && sb && sb->bound_k)
      MCLST_CUDA(cudaMemsetAsync(sb->bound_k, 0xff, (size_t)n_query * 4, st));
    if ((stages & 2) && !(stages & 4) && sb && sb->bound_part)
      MCLST_CUDA(cudaMemsetAsync(sb->bound_part, 0xff, (size_t)n_query * 4, st));
    if (!(stages & 4) || n_query == 0) return 0;
    MCLST_CUDA(cudaMemsetAsync(w.counters, 0, 256, st));
    prof_mark(st, "row_norms");
    if ((rc = launch_row_norms(bank, n_bank, ld_bank, dim, w.bank_nrm, st))) return rc;
    if ((rc = launch_row_norms(query, n_query, ld_query, dim, w.q_nrm, st))) return rc;
    prof_mark(st, "exact_topk");
    rc = launch_exact_topk(bank, n_bank, ld_bank, w.bank_nrm, query, ld_query, w.q_nrm, dim,
                           nullptr, nullptr, (int)n_query, n_query, top_k, index_offset, w.scratch,
                           out_indices, out_values, st);
    if (!rc && out_distances)
      rc = launch_neighbor_distances(bank, n_bank, ld_bank, query, n_query, ld_query, dim, out_indices,
                                     top_k, index_offset, dist_p, out_distances, nullptr, nullptr, st);
    prof_mark(st, "end");
    return rc;
  }
  const TcWorkspace& t = w.tc;
  if (stages & 1) {
    prof_mark(st, "pack_rows");
    if (!packed) {
      MCLST_CUDA(cudaMemsetAsync(t.stats, 0, 8 * sizeof(uint32_t), st));
      if ((rc = launch_pack_rows(bank, n_bank, t.n_pad, ld_bank, dim, t.nkb, t.bpack, t.b_nrm,
                                 t.b_resid, t.stats, st))) return rc;
    }
    if (n_query == 0) { prof_mark(st, "end"); return 0; }
    MCLST_CUDA(cudaMemsetAsync(w.counters, 0, 256, st));
    MCLST_CUDA(cudaMemsetAsync(t.stats + 8, 0, 8 * sizeof(uint32_t), st));
    if ((rc = launch_pack_rows(query, n_query, t.q_pad, ld_query, dim, t.nkb, t.qpack, t.q_nrm,
                               t.q_resid, t.stats + 8, st))) return rc;
    if (stages == 1) {          // seed pass alone; the main pass follows in a second call
      prof_mark(st, "sim_seed");
      if ((rc = launch_sim_topk(t, n_bank, n_query, top_k, st, 1, sb))) return rc;
      prof_mark(st, "end");
      return 0;
    }
  }
  if (n_query == 0) return 0;
  if (stages & 2) {
    prof_mark(st, "sim_topk");
    if ((rc = launch_sim_topk(t, n_bank, n_query, top_k, st, (stages & 1) ? 0 : 2, sb))) return rc;
    if (!(stages & 4)) {
      if (sb && sb->bound_k && (rc = launch_export_bound(t, n_query, top_k, sb->bound_k, sb->k_part, sb->bound_part, st))) return rc;
      prof_mark(st, "end");
      return 0;
    }
  } else if (sb && sb->ext_bound) {
    if ((rc = launch_apply_bound(t, n_query, sb->ext_bound, st))) return rc;
  }
  prof_mark(st, "rerank");
  if ((rc = launch_rerank(t, bank, n_bank, ld_bank, query, n_query, ld_query, dim, top_k,
                          index_offset, out_indices, out_values, out_distances, dist_p, w.counters,
                          st, sb && sb->ext_bound))) return rc;
  prof_mark(st, "exact_fallback");
  rc = launch_exact_topk(bank, n_bank, ld_bank, w.bank_nrm, query, ld_query, w.q_nrm, dim,
                         t.fb_list, w.counters, 0, n_query, top_k, index_offset, w.scratch,
                         out_indices, out_values, st);
  if (!rc && out_distances)      // rows the exact path recomputed: their distances too
    rc = launch_neighbor_distances(bank, n_bank, ld_bank, query, n_query, ld_query, dim, out_indices,
                                   top_k, index_offset, dist_p, out_distances, t.fb_list, w.counters, st);
  prof_mark(st, "end");
  return rc;
}

extern "C" int mclst_find_matches_dist(const float* bank, int64_t n_bank, int64_t ld_bank,
                                       const float* query, int64_t n_query, int64_t ld_query,
                                       int dim, int top_k, int64_t index_offset,
                                       int64_t* out_indices, float* out_values,
                                       float* out_distances, int dist_p, void* workspace,
                                       size_t workspace_bytes, int flags, mclst_stream_t stream) {
  if (n_query == 0 && n_bank >= 0 && !(flags & MCLST_FM_BANK_PACKED)) return 0;
  return find_matches_stages(7, bank, n_bank, ld_bank, query, n_query, ld_query, dim, top_k, index_offset,
                             out_indices, out_values, out_distances, dist_p, nullptr, workspace,
                             workspace_bytes, flags, (cudaStream_t)stream);
}

extern "C" int mclst_find_matches_pack_bank(const float* bank, int64_t n_bank, int64_t ld_bank, int dim,
                                            int top_k, void* workspace, size_t workspace_bytes,
                                            mclst_stream_t stream) {
  return find_matches_stages(1, bank, n_bank, ld_bank, nullptr, 0, dim, dim, top_k, 0, nullptr, nullptr,
                             nullptr, 2, nullptr, workspace, workspace_bytes, 0, (cudaStream_t)stream);
}

extern "C" int mclst_find_matches_seed(const float* bank, int64_t n_bank, int64_t ld_bank,
                                       const float* query, int64_t n_query, int64_t ld_query, int dim,
                                       int top_k, int k_part, float* bound_k, float* bound_part,
                                       void* workspace, size_t workspace_bytes, int flags,
                                       mclst_stream_t stream) {
  MCLST_REQUIRE(k_part >= 1 && k_part <= top_k, MCLST_ERR_INVALID, "find_matches_seed: k_part");
  SeedBounds sb{k_part, bound_k, bound_part, nullptr};
  return find_matches_stages(1, bank, n_bank, ld_bank, query, n_query, ld_query, dim, top_k, 0, nullptr,
                             nullptr, nullptr, 2, &sb, workspace, workspace_bytes, flags,
                             (cudaStream_t)stream);
}

extern "C" int mclst_find_matches_main(const float* bank, int64_t n_bank, int64_t ld_bank,
                                       const float* query, int64_t n_query, int64_t ld_query, int dim,
                                       int top_k, int64_t index_offset, int64_t* out_indices,
                                       float* out_values, float* out_distances, int dist_p,
                                       const float* ext_bound, void* workspace, size_t workspace_bytes,
                                       int flags, mclst_stream_t stream) {
  if (n_query == 0) return 0;
  SeedBounds sb{1, nullptr, nullptr, ext_bound};
  return find_matches_stages(6, bank, n_bank, ld_bank, query, n_query, ld_query, dim, top_k, index_offset,
                             out_indices, out_values, out_distances, dist_p, &sb, workspace,
                             workspace_bytes, flags, (cudaStream_t)stream);
}

extern "C" int mclst_find_matches_candidates(const float* bank, int64_t n_bank, int64_t ld_bank,
                                             const float* query, int64_t n_query, int64_t ld_query,
                                             int dim, int top_k, int k_part, const float* ext_bound,
                                             float* bound_out, float* bound_part_out, void* workspace,
                                             size_t workspace_bytes, int flags, mclst_stream_t stream) {
  if (n_query == 0) return 0;
  MCLST_REQUIRE(bound_out, MCLST_ERR_INVALID, "find_matches_candidates: null bound_out");
  SeedBounds sb{k_part, bound_out, bound_part_out, ext_bound};
  return find_matches_stages(2, bank, n_bank, ld_bank, query, n_query, ld_query, dim, top_k, 0, nullptr,
                             nullptr, nullptr, 2, &sb, workspace, workspace_bytes, flags,
                             (cudaStream_t)stream);
}

extern "C" int mclst_find_matches_finish(const float* bank, int64_t n_bank, int64_t ld_bank,
                                         const float* query, int64_t n_query, int64_t ld_query, int dim,
                                         int top_k, int64_t index_offset, int64_t* out_indices,
                                         float* out_values, float* out_distances, int dist_p,
                                         const float* ext_bound, void* workspace, size_t workspace_bytes,
                                         int flags, mclst_stream_t stream) {
  if (n_query == 0) return 0;
  SeedBounds sb{1, nullptr, nullptr, ext_bound};
  return find_matches_stages(4, bank, n_bank, ld_bank, query, n_query, ld_query, dim, top_k, index_offset,
                             out_indices, out_values, out_distances, dist_p, &sb, workspace,
                             workspace_bytes, flags, (cudaStream_t)stream);
}

// ---- the whole fold-loop body in one call ------------------------------------------------------
// find_matches (+ neighbour distances) and the weighted expression average.  Very large query
// sets go through in blocks (bounded workspace): the candidate pass, re-rank and exact fallback of
// block b run on `stream`, the HBM-bound average of block b on an internal side stream, so that it
// fills whatever the candidate pass of block b + 1 leaves free, and is joined back at the end.
namespace mclst {
struct SideStream {
  cudaStream_t st = nullptr;
  std::vector<cudaEvent_t> ev;
  size_t next = 0;
  cudaEvent_t event() {                       // round-robin over a small pool (re-recording an event
    if (ev.size() < 16) {                     // whose earlier waits are already enqueued is fine)
      cudaEvent_t e;
      if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return nullptr;
      ev.push_back(e);
      return e;
    }
    return ev[next++ % ev.size()];
  }
};
static std::mutex g_side_mu;
static SideStream g_side[64];

int side_fork(cudaStream_t st, cudaStream_t* side_out) {
  int dev = 0;
  MCLST_CUDA(cudaGetDevice(&dev));
  MCLST_REQUIRE(dev >= 0 && dev < 64, MCLST_ERR_DEVICE, "side stream: device ordinal %d", dev);
  std::lock_guard<std::mutex> lk(g_side_mu);
  SideStream& s = g_side[dev];
  if (!s.st) MCLST_CUDA(cudaStreamCreateWithFlags(&s.st, cudaStreamNonBlocking));
  cudaEvent_t e = s.event();
  MCLST_REQUIRE(e, MCLST_ERR_DEVICE, "side stream: event creation failed");
  MCLST_CUDA(cudaEventRecord(e, st));
  MCLST_CUDA(cudaStreamWaitEvent(s.st, e, 0));
  *side_out = s.st;
  return 0;
}

int side_join(cudaStream_t st) {
  int dev = 0;
  MCLST_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(g_side_mu);
  SideStream& s = g_side[dev];
  MCLST_REQUIRE(s.st, MCLST_ERR_INVALID, "side stream: join without fork");
  cudaEvent_t e = s.event();
  MCLST_REQUIRE(e, MCLST_ERR_DEVICE, "side stream: event creation failed");
  MCLST_CUDA(cudaEventRecord(e, s.st));
  MCLST_CUDA(cudaStreamWaitEvent(st, e, 0));
  return 0;
}

// path counters of a blocked call: every block resets the four counters at the head of the
// workspace (the exact-fallback list is indexed by one of them), so the totals are kept aside and
// written back after the last block.  mode 0: clear totals, 1: totals += counters, 2: counters = totals
__global__ void counters_fold_kernel(int* counters, int* totals, int mode) {
  const int i = threadIdx.x;
  if (i >= 4) return;
  if (mode == 0) totals[i] = 0;
  else if (mode == 1) totals[i] += counters[i];
  else counters[i] = totals[i];
}

// Measured at cfg4 (65 536 queries): blocks of one lane round gain nothing -- the persistent
// candidate kernel owns the whole register file of every SM (10 warps are allocated as 12 x 168
// registers), so the average of a block cannot run beside it and only moves to the gaps, while four
// seed passes instead of one cost 0.4 ms (33.5 vs 33.1 ms per step).  With the candidate kernel capped
// at 144 / 128 registers (__maxnreg__) the average does run underneath (1.8 ms of overlap measured),
// but the cap costs the candidate pass 1.1 / 3.0 ms: 29.7 / 31.5 ms against 29.5 ms unblocked.
// Blocking therefore only bounds the workspace of very large query sets (candidate buffers: 8 KiB
// per query).
static int64_t retrieve_block_rows(int64_t n_query) {
  const int64_t round = 128ll * sm_count();
  return n_query > 8 * round ? 4 * round : n_query;
}
}  // namespace mclst

extern "C" int mclst_retrieve_workspace_bytes(int64_t n_bank, int64_t n_query, int dim, int top_k, int flags,
                                              size_t* bytes) {
  MCLST_REQUIRE(bytes, MCLST_ERR_INVALID, "retrieve_workspace_bytes: null pointer");
  MCLST_REQUIRE(n_bank >= 0 && n_query >= 0 && dim >= 1 && top_k >= 1, MCLST_ERR_INVALID,
                "retrieve_workspace_bytes: bad shape");
  const size_t fm = carve_fm(nullptr, 0, n_bank, retrieve_block_rows(n_query), dim, top_k, flags).bytes;
  *bytes = align_up(fm, 256) + align_up((size_t)n_query * top_k * sizeof(float), 256) + 256 /*counter totals*/;
  return 0;
}

extern "C" int mclst_weighted_average(const float* spot_key, int64_t n_bank, int64_t ld_key,
                                      const void* expression_key, int64_t ld_expr, int genes,
                                      int expr_is_f64, const float* image_query, int64_t n_query,
                                      int64_t ld_query, int dim, const int64_t* indices,
                                      const float* values, const float* distances, int top_k,
                                      int64_t index_offset, int weight_mode, void* out_emb,
                                      void* out_expr, int out_is_f64, mclst_stream_t stream);

extern "C" int mclst_retrieve(const float* bank, int64_t n_bank, int64_t ld_bank, const void* expression_key,
                              int64_t ld_expr, int genes, int expr_is_f64, const float* query,
                              int64_t n_query, int64_t ld_query, int dim, int top_k, int weight_mode,
                              int64_t* out_indices, float* out_values, void* out_emb, void* out_expr,
                              int out_is_f64, void* workspace, size_t workspace_bytes, int flags,
                              mclst_stream_t stream) {
  MCLST_REQUIRE(bank && expression_key && workspace && out_indices && out_expr && (query || n_query == 0),
                MCLST_ERR_INVALID, "retrieve: null pointer");
  MCLST_REQUIRE(weight_mode >= 0 && weight_mode <= MCLST_W_BLEEP_EXP, MCLST_ERR_INVALID,
                "retrieve: bad weight mode %d", weight_mode);
  MCLST_REQUIRE(weight_mode != MCLST_W_SIMILARITY || out_values, MCLST_ERR_INVALID,
                "retrieve: similarity weights need out_values");
  if (n_query == 0) return 0;
  size_t need = 0;
  int rc = mclst_retrieve_workspace_bytes(n_bank, n_query, dim, top_k, flags, &need);
  if (rc) return rc;
  MCLST_REQUIRE(need <= workspace_bytes, MCLST_ERR_WORKSPACE, "retrieve: workspace %zu < %zu", workspace_bytes, need);
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t QB = retrieve_block_rows(n_query);
  const size_t fm_bytes = align_up(carve_fm(nullptr, 0, n_bank, QB, dim, top_k, flags).bytes, 256);
  const bool need_dist = weight_mode == MCLST_W_INV_SQ_L1 || weight_mode == MCLST_W_INV_SQ_L2 ||
                         weight_mode == MCLST_W_BLEEP_EXP;
  float* dist = need_dist ? reinterpret_cast<float*>(static_cast<char*>(workspace) + fm_bytes) : nullptr;
  const int dist_p = weight_mode == MCLST_W_INV_SQ_L1 ? 1 : 2;
  int* counters = static_cast<int*>(workspace);
  int* totals = reinterpret_cast<int*>(static_cast<char*>(workspace) + fm_bytes +
                                       align_up((size_t)n_query * top_k * sizeof(float), 256));
  const size_t esz = expr_is_f64 ? 8 : 4, osz = out_is_f64 ? 8 : 4;
  (void)esz;
  const bool overlap = QB < n_query;
  if (overlap) counters_fold_kernel<<<1, 32, 0, st>>>(counters, totals, 0);
  for (int64_t q0 = 0, b = 0; q0 < n_query; q0 += QB, ++b) {
    const int64_t nq = std::min(QB, n_query - q0);
    // the bank is packed by the first block; later blocks find its image at the head of the workspace
    const int f = flags | (b > 0 ? MCLST_FM_BANK_PACKED : 0);
    const bool tc = tc_eligible(n_bank, dim, top_k, f);
    rc = find_matches_stages(7, bank, n_bank, ld_bank, query + q0 * ld_query, nq, ld_query, dim, top_k, 0,
                             out_indices + q0 * top_k, out_values ? out_values + q0 * top_k : nullptr,
                             dist ? dist + q0 * top_k : nullptr, dist_p, nullptr, workspace, fm_bytes,
                             tc ? f : (f & ~MCLST_FM_BANK_PACKED), st);
    if (rc) return rc;
    cudaStream_t as = st;
    if (overlap) {
      counters_fold_kernel<<<1, 32, 0, st>>>(counters, totals, 1);
      if ((rc = side_fork(st, &as))) return rc;
    }
    rc = mclst_weighted_average(bank, n_bank, ld_bank, expression_key, ld_expr, genes, expr_is_f64,
                                query + q0 * ld_query, nq, ld_query, dim, out_indices + q0 * top_k,
                                out_values ? out_values + q0 * top_k : nullptr, dist ? dist + q0 * top_k : nullptr,
                                top_k, 0, weight_mode,
                                out_emb ? static_cast<char*>(out_emb) + (size_t)q0 * dim * osz : nullptr,
                                static_cast<char*>(out_expr) + (size_t)q0 * genes * osz, out_is_f64,
                                (mclst_stream_t)as);
    if (rc) return rc;
  }
  if (overlap) {                                         // join: `stream` continues after the last average
    counters_fold_kernel<<<1, 32, 0, st>>>(counters, totals, 2);
    MCLST_LAUNCH_CHECK();
    if ((rc = side_join(st))) return rc;
  }
  return 0;
}

// Testing aid: the raw tensor-core similarities the candidate pass sees (fp16-rounded
// normalised operands, fp32 accumulation), written to out [n_query, ld_out].
extern "C" int mclst_debug_similarity(const float* bank, int64_t n_bank, int64_t ld_bank,
                                      const float* query, int64_t n_query, int64_t ld_query,
                                      int dim, float* out, int64_t ld_out, void* workspace,
                                      size_t workspace_bytes, mclst_stream_t stream) {
  MCLST_REQUIRE(bank && query && out && workspace, MCLST_ERR_INVALID, "debug_similarity: null");
  MCLST_REQUIRE(dim >= 1 && dim <= TC_MAX_DIM, MCLST_ERR_UNSUPPORTED, "debug_similarity: dim %d > %d", dim,
                TC_MAX_DIM);
  cudaStream_t st = (cudaStream_t)stream;
  FmWorkspace w = carve_fm(workspace, workspace_bytes, n_bank, n_query, dim, 1, 0);
  MCLST_REQUIRE(w.use_tc && w.bytes <= workspace_bytes, MCLST_ERR_WORKSPACE, "debug_similarity: ws");
  const TcWorkspace& t = w.tc;
  int rc;
  MCLST_CUDA(cudaMemsetAsync(t.stats, 0, 16 * sizeof(uint32_t), st));
  if ((rc = launch_pack_rows(bank, n_bank, t.n_pad, ld_bank, dim, t.nkb, t.bpack, t.b_nrm,
                             t.b_resid, t.stats, st))) return rc;
  if ((rc = launch_pack_rows(query, n_query, t.q_pad, ld_query, dim, t.nkb, t.qpack, t.q_nrm,
                             t.q_resid, t.stats + 8, st))) return rc;
  return launch_sim_dump(t, n_bank, n_query, out, ld_out, st);
}
