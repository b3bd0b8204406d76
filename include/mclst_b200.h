/*
 * mclst_b200.h -- C-ABI of libmclst_b200.so: the B200 (sm_100a) kernels behind the
 * mclSTExp contrastive-alignment + retrieval hot path.
 *
 * The reference (ZhicengShi/mclSTExp) is pure Python/PyTorch and has NO FFI layer of its
 * own (SURVEY.md section 8b); each entry point below names the reference lines whose
 * arithmetic it replaces, and INTEGRATION.md shows the ctypes stub a maintainer adds to
 * model.py / evel_*.py.  Conventions:
 *
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless the
 *     parameter name ends in _host;
 *   - the caller owns every buffer (inputs, outputs, workspace); a *_workspace_bytes()
 *     query precedes each op that needs scratch; the library keeps no tensor state;
 *   - every call is asynchronous on `stream` (a cudaStream_t) and never synchronises;
 *   - return value: 0 = ok, negative = MCLST_ERR_*, positive = cudaError_t;
 *     mclst_last_error() returns a thread-local message for the last failure;
 *   - matrices are row-major float32 with an explicit leading dimension (elements).
 */
#ifndef MCLST_B200_H
#define MCLST_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* mclst_stream_t; /* cudaStream_t */

enum {
  MCLST_OK = 0,
  MCLST_ERR_INVALID = -1,     /* bad argument (null pointer, k > N, misaligned, ...) */
  MCLST_ERR_WORKSPACE = -2,   /* workspace too small */
  MCLST_ERR_UNSUPPORTED = -3, /* shape outside what the kernels are built for */
  MCLST_ERR_DEVICE = -4       /* not an sm_100 device */
};

/* weight modes of the top-k expression average */
enum {
  MCLST_W_INV_SQ_L1 = 0, /* evel_her2st.py:178-184  (ord=1)                          */
  MCLST_W_INV_SQ_L2 = 1, /* evel_visium.py:197-200, evel_cscc.py:209-211             */
  MCLST_W_SIMILARITY = 2,/* evel_cscc.py:201 (commented variant): value / sum(value) */
  MCLST_W_UNIFORM = 3,   /* BLEEP_inference.ipynb cell 5 "average" / "simple" (k=1)  */
  MCLST_W_BLEEP_EXP = 4  /* BLEEP_inference.ipynb cell 5 "weighted_average"          */
};

/* flags of mclst_find_matches / mclst_retrieve */
enum {
  MCLST_FM_DEFAULT = 0,
  MCLST_FM_EXACT_ONLY = 1, /* skip the tensor-core candidate pass, brute-force every query */
  MCLST_FM_NO_SPECULATION = 4, /* start the running top-k thresholds from the guaranteed seed only
                              (default: a speculative, verified one -- csrc/sim_topk.cu spec_rank) */
  MCLST_FM_BANK_PACKED = 2 /* the workspace already holds this bank's packed image (an earlier
                              mclst_find_matches_pack_bank / _seed / find_matches call on the same
                              workspace with the same bank, n_bank, dim and top_k): skip the bank pass */
};

/* contrastive-loss target modes */
enum {
  MCLST_T_EYE = 0,      /* model.py:242-247                                        */
  MCLST_T_SOFT_DIV = 1, /* baselines/Bleep/models.py:34-43   (.../2/T)             */
  MCLST_T_SOFT_MUL = 2  /* baselines/Bleep/models.py:70-79   (.../2*T)             */
};

int mclst_version(void);
const char* mclst_last_error(void);
/* sm count / compute capability of the current device; MCLST_ERR_DEVICE if not sm_100 */
int mclst_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* number of kernels this library has launched since load (claim for bench.py gpu_launches) */
int64_t mclst_launch_count(void);
/* mclst_find_matches keeps counters at the head of its workspace (device).  This copies them
 * out (synchronises `stream`): [0] queries resolved by the tensor-core candidate path,
 * [1] queries recomputed by the exact brute-force path. */
int mclst_read_counters(const void* workspace, int64_t counters_host[4], mclst_stream_t stream);

/* Per-kernel CUDA-event trace for bench.py's roofline block.  enable(1) starts recording
 * one event per internal kernel launch on the launching stream; collect() synchronises and
 * returns (name, milliseconds) per kernel since the last collect.  names: 48-byte records. */
int mclst_profile_enable(int on);
int mclst_profile_collect(char* names_out, float* ms_out, int cap, int* n);

/* ---------------------------------------------------------------- retrieval ---------- */

/* find_matches  (evel_her2st.py:74-84, evel_visium.py:94-104, evel_cscc.py:74-84).
 * L2-normalise bank rows and query rows (F.normalize, eps 1e-12), rank every bank row by
 * cosine similarity per query and return the top_k, sorted by (similarity descending,
 * index ascending).  out_indices [n_query, top_k] int64 (torch.topk's dtype), each index
 * + index_offset (bank shards).  out_values (nullable) [n_query, top_k] float32 are the
 * similarities the cSCC flavour returns.  Any dim works; the output is always the exact one.
 * Calls with dim <= 512, top_k <= 896 and top_k <= n_bank (mclst_find_matches_tc_eligible) run
 * the tensor-core candidate pass plus an exact re-rank; all others, and MCLST_FM_EXACT_ONLY,
 * brute-force every query in float64. */
int mclst_find_matches_workspace_bytes(int64_t n_bank, int64_t n_query, int dim, int top_k,
                                       int flags, size_t* bytes);
int mclst_find_matches(const float* bank, int64_t n_bank, int64_t ld_bank,
                       const float* query, int64_t n_query, int64_t ld_query,
                       int dim, int top_k, int64_t index_offset,
                       int64_t* out_indices, float* out_values,
                       void* workspace, size_t workspace_bytes, int flags,
                       mclst_stream_t stream);

/* Same, additionally returning out_distances [n_query, top_k] float32: the L1 (dist_p = 1,
 * evel_her2st.py:178) or L2 (dist_p = 2, evel_visium.py:197) norm of (bank row - query) on the
 * UN-normalised vectors for every winner -- the quantity the weighted-average loop needs --
 * computed while the re-rank has the rows in registers instead of gathering them again. */
int mclst_find_matches_dist(const float* bank, int64_t n_bank, int64_t ld_bank,
                            const float* query, int64_t n_query, int64_t ld_query,
                            int dim, int top_k, int64_t index_offset,
                            int64_t* out_indices, float* out_values, float* out_distances,
                            int dist_p, void* workspace, size_t workspace_bytes, int flags,
                            mclst_stream_t stream);

/* Staged form of mclst_find_matches_dist, for
 *  (a) bank shards (one per GPU, SURVEY.md 8e): every shard runs the SEED pass, the ranks exchange
 *      a lower bound of the exact GLOBAL k-th best score per query, and every shard's MAIN pass
 *      filters against it instead of converging its own threshold from scratch;
 *  (b) a bank kept resident on the device (the serving form of the fold loop, and the hand-off
 *      from the bank build, evel_her2st.py:44-71,116-117): _pack_bank writes the normalised fp16
 *      operand image, float64 norms and rounding residuals of the bank rows into the workspace
 *      once; later _seed / find_matches calls pass MCLST_FM_BANK_PACKED and only pack the queries
 *      (the bank-derived part of the workspace does not depend on n_query; size the workspace with
 *      mclst_find_matches_workspace_bytes for the largest query batch).
 * _seed:  bound_k[q] (nullable) <= the exact score of at least top_k rows of THIS bank;
 *         bound_part[q] (nullable) likewise for k_part <= top_k rows; -inf or NaN = nothing known.
 *         For R homogeneous shards min over shards of bound_part with k_part = ceil(top_k / R) is a
 *         valid (and much tighter) bound of the global k-th best, as is max over shards of bound_k.
 * _main:  must follow _seed on the same workspace and stream order.  ext_bound (nullable) [n_query]:
 *         rows provably below it are dropped, so a shard may return FEWER than top_k rows for a
 *         query: the tail of its list is padded with (value -inf, index 0x7fffffff, distance +inf),
 *         which loses every mclst_merge_topk comparison.
 * _candidates + _finish: _main in two halves with a second, much tighter exchange in between.
 *         _candidates runs the tensor-core candidate pass (against ext_bound when given) and
 *         writes, from the candidates it kept, bound_out[q] / bound_part_out[q] (nullable): lower
 *         bounds of this shard's exact top_k-th / k_part-th best score.  max over shards of
 *         bound_out and min over shards of bound_part_out (k_part = ceil(top_k / shards)) both
 *         bound the global top_k-th best; passed to _finish, the larger lets every shard re-rank
 *         (exactly) only the candidates that can still be among the global winners -- about
 *         (top_k + band) / shards rows instead of top_k + band.  Pass _finish a bound at least as
 *         tight as the one _candidates got. */
int mclst_find_matches_pack_bank(const float* bank, int64_t n_bank, int64_t ld_bank, int dim,
                                 int top_k, void* workspace, size_t workspace_bytes,
                                 mclst_stream_t stream);
int mclst_find_matches_seed(const float* bank, int64_t n_bank, int64_t ld_bank,
                            const float* query, int64_t n_query, int64_t ld_query, int dim,
                            int top_k, int k_part, float* bound_k, float* bound_part,
                            void* workspace, size_t workspace_bytes, int flags,
                            mclst_stream_t stream);
int mclst_find_matches_main(const float* bank, int64_t n_bank, int64_t ld_bank,
                            const float* query, int64_t n_query, int64_t ld_query, int dim,
                            int top_k, int64_t index_offset, int64_t* out_indices,
                            float* out_values, float* out_distances, int dist_p,
                            const float* ext_bound, void* workspace, size_t workspace_bytes,
                            int flags, mclst_stream_t stream);

int mclst_find_matches_candidates(const float* bank, int64_t n_bank, int64_t ld_bank,
                                  const float* query, int64_t n_query, int64_t ld_query, int dim,
                                  int top_k, int k_part, const float* ext_bound, float* bound_out,
                                  float* bound_part_out, void* workspace, size_t workspace_bytes,
                                  int flags, mclst_stream_t stream);
int mclst_find_matches_finish(const float* bank, int64_t n_bank, int64_t ld_bank,
                              const float* query, int64_t n_query, int64_t ld_query, int dim,
                              int top_k, int64_t index_offset, int64_t* out_indices,
                              float* out_values, float* out_distances, int dist_p,
                              const float* ext_bound, void* workspace, size_t workspace_bytes,
                              int flags, mclst_stream_t stream);

/* 1 if a find_matches call of this shape and flags runs the tensor-core candidate pass, 0 if it
 * brute-forces every query: !(flags & MCLST_FM_EXACT_ONLY) && 1 <= dim <= 512 && top_k <= 896
 * && top_k <= n_bank.  MCLST_FM_BANK_PACKED needs it.  Host only, no device needed. */
int mclst_find_matches_tc_eligible(int64_t n_bank, int dim, int top_k, int flags);

/* Testing aid: the raw similarities of the tensor-core candidate pass (fp16-rounded
 * normalised operands, fp32 accumulation) written to out [n_query, ld_out]; dim <= 512;
 * workspace as for mclst_find_matches with top_k = 1.  Not part of the reference surface. */
int mclst_debug_similarity(const float* bank, int64_t n_bank, int64_t ld_bank,
                           const float* query, int64_t n_query, int64_t ld_query, int dim,
                           float* out, int64_t ld_out, void* workspace, size_t workspace_bytes,
                           mclst_stream_t stream);

/* Testing aid (host only): the rank j <= top_k of the sample value the speculative seed threshold
 * starts from when a fraction `sampled_fraction` of the bank tiles is sampled: the smallest j with
 * P(Binomial(top_k - 1, sampled_fraction) >= j) < 1e-7 (csrc/sim_topk.cu, spec_rank). */
int mclst_debug_spec_rank(int top_k, double sampled_fraction);

/* Testing aid (host only, no device needed): the work decomposition of the persistent top-k
 * kernel for query_blocks x bank_tiles on `lanes` SMs with at most max_slots candidate streams
 * per query block.  Writes up to max_units records {lane, query_block, tile_begin, tile_end,
 * slot} (5 ints each) to units and their number to *n_units; *slots = streams per query block.
 * Not part of the reference surface. */
int mclst_debug_lane_plan(int64_t query_blocks, int64_t bank_tiles, int lanes, int max_slots,
                          int* units, int64_t max_units, int64_t* n_units, int* slots);

/* Testing aid (host only, no device needed): the tile kernel mclst_matmul's packed fp16 route runs
 * for an M x N output with `batch` products, on the current device's SM count (148 without a
 * device): *cluster = 2 for CTA pairs that share B (128 x 256 tiles) or 1, *width = the tile width
 * 256, 128 or 64.  Honours MCLST_GEMM_CLUSTER like the launch does.  Not part of the reference
 * surface. */
int mclst_debug_gemm_variant(int64_t M, int64_t N, int batch, int* cluster, int* width);

/* The whole fold-loop body (evel_her2st.py:174-187: find_matches, then the per-query loop) in ONE
 * call on device-resident arrays: out_indices [n_query, top_k] int64, out_values (nullable unless
 * MCLST_W_SIMILARITY) [n_query, top_k] float32, out_emb (nullable) [n_query, dim], out_expr
 * [n_query, genes] (float32, or float64 when out_is_f64).  Query sets beyond eight rounds of the
 * persistent top-k kernel (8 x 128 x SM count rows) go through in blocks, which bounds the workspace;
 * the expression average of a block then runs on an internal side stream next to the top-k pass of
 * the following block and is joined back into `stream` before the call returns (stream-ordered
 * like every other entry).  flags: MCLST_FM_*; with
 * MCLST_FM_BANK_PACKED the workspace already holds this bank's packed image
 * (mclst_find_matches_pack_bank on a workspace of mclst_retrieve_workspace_bytes). */
int mclst_retrieve_workspace_bytes(int64_t n_bank, int64_t n_query, int dim, int top_k, int flags,
                                   size_t* bytes);
int mclst_retrieve(const float* bank, int64_t n_bank, int64_t ld_bank, const void* expression_key,
                   int64_t ld_expr, int genes, int expr_is_f64, const float* query, int64_t n_query,
                   int64_t ld_query, int dim, int top_k, int weight_mode, int64_t* out_indices,
                   float* out_values, void* out_emb, void* out_expr, int out_is_f64, void* workspace,
                   size_t workspace_bytes, int flags, mclst_stream_t stream);

/* The per-query loop evel_her2st.py:175-187 / evel_visium.py:194-205 /
 * evel_cscc.py:198-215 / BLEEP_inference.ipynb cell 5: weights from the UN-normalised
 * spot_key rows selected by `indices` and the query, then the weighted average of those
 * spot_key rows (out_emb, nullable) and of the matching expression_key rows (out_expr).
 * expression_key is [n_bank, genes] float32 (expr_is_f64 = 0) or float64 (= 1); outputs
 * are float64 (out_is_f64 = 1, the reference's np.zeros dtype) or float32.
 * indices [n_query, top_k] int64 are global row numbers (local row = index - index_offset).
 * values (only MCLST_W_SIMILARITY) [n_query, top_k] float32.  distances (nullable)
 * [n_query, top_k] float32: neighbour distances already known (mclst_find_matches_dist); when
 * null they are computed here from the gathered rows. */
int mclst_weighted_average(const float* spot_key, int64_t n_bank, int64_t ld_key,
                           const void* expression_key, int64_t ld_expr, int genes, int expr_is_f64,
                           const float* image_query, int64_t n_query, int64_t ld_query, int dim,
                           const int64_t* indices, const float* values, const float* distances,
                           int top_k, int64_t index_offset, int weight_mode,
                           void* out_emb, void* out_expr, int out_is_f64,
                           mclst_stream_t stream);

/* Partial (sharded-bank) form of the same loop: writes UN-normalised weights
 * w [n_query, top_k] float32 for the winners this shard owns (index in
 * [index_offset, index_offset + n_bank), others 0) and accumulates nothing.  Used by the
 * multi-GPU merge; see mclstexp_b200/retrieval.py. */
int mclst_neighbor_distances(const float* spot_key, int64_t n_bank, int64_t ld_key,
                             const float* image_query, int64_t n_query, int64_t ld_query, int dim,
                             const int64_t* indices, int top_k, int64_t index_offset, int p,
                             float* out_dist, mclst_stream_t stream);
int mclst_weighted_gather(const void* expression_key, int64_t n_bank, int64_t ld_expr, int genes,
                          int expr_is_f64, const int64_t* indices, const float* weights,
                          int64_t n_query, int top_k, int64_t index_offset,
                          float* out_partial /* [n_query, genes] float32, overwritten */,
                          mclst_stream_t stream);

/* Row-sharded form (embedding all-gather over NVLink, SURVEY.md section 8e): spot_emb /
 * image_emb are the ALL-GATHERED [batch, dim] embeddings; this rank owns the rows
 * [row0, row0 + rows) (row0 a multiple of 128).  `stats` is a caller-owned device block
 * [MCLST_LOSS_STAT_ROWS][batch] float32 (rl, cl, za, wbar, cs, diag, rl_lo, cl_lo, za_lo: the three
 * log-sum-exp statistics are float PAIRS hi + lo) whose local slices each phase fills and
 * which the caller all-gathers between phases:
 *   phase 1 packs the operands and writes rl, cl, za (+ their lo parts), diag of the local rows;
 *   phase 2 (after gathering those) writes wbar, cs of the local rows (soft targets);
 *   phase 3 (after gathering wbar, cs) writes this rank's additive loss contribution to
 *           *loss_out and, if d_spot/d_image are given, the gradients of the LOCAL rows
 *           ([rows, dim]); no gradient exchange is needed afterwards.
 * The same workspace must be passed to all three phases. */
#define MCLST_LOSS_STAT_ROWS 9
int mclst_contrastive_loss_phase(const float* spot_emb, int64_t ld_s, const float* image_emb,
                                 int64_t ld_i, int batch, int dim, float temperature, int target_mode,
                                 int64_t row0, int64_t rows, int phase, float* stats, float* loss_out,
                                 float* d_spot, int64_t ld_ds, float* d_image, int64_t ld_di,
                                 void* workspace, size_t workspace_bytes, mclst_stream_t stream);

/* Sharded-bank merge (no reference counterpart: the reference is single-process).  `values`,
 * `indices`, `distances` are the per-shard results gathered as [n_lists, n_query, top_k];
 * the output is the global top_k by (value descending, index ascending) with the distances
 * carried along (distances / out_distances may both be null). */
int mclst_merge_topk(const float* values, const int64_t* indices, const float* distances,
                     int n_lists, int64_t n_query, int top_k, float* out_values,
                     int64_t* out_indices, float* out_distances, mclst_stream_t stream);
/* Normalised weights [n_query, top_k] from neighbour distances (L1 for MCLST_W_INV_SQ_L1, L2
 * otherwise) or similarities -- the weight formulas of mclst_weighted_average. */
int mclst_neighbor_weights(const float* distances, const float* values, int64_t n_query, int top_k,
                           int weight_mode, float* out_weights, mclst_stream_t stream);

/* ---------------------------------------------------------------- evaluation metrics ---- */

/* Per-gene statistics of the predicted vs true expression matrices ([n_spots, genes], float32
 * or float64): mean of the truth (top-50 HEG selection, evel_her2st.py:201-205), Pearson r
 * (utils.py:52-65 get_R / scipy pearsonr; NaN for a constant column), and the per-gene sums of
 * squared and absolute errors (sklearn MSE / MAE at evel_her2st.py:214-221 are their totals over
 * n_spots * genes).  All outputs float64 [genes]; scratch from mclst_gene_metrics_scratch_doubles. */
int mclst_gene_metrics_scratch_doubles(int genes, size_t* n);
int mclst_gene_metrics(const void* truth, int64_t ld_true, int true_is_f64, const void* pred,
                       int64_t ld_pred, int pred_is_f64, int64_t n_spots, int genes,
                       double* mean_true, double* pcc, double* sq_err, double* abs_err,
                       double* scratch, mclst_stream_t stream);

/* ---------------------------------------------------------------- contrastive loss ------ */

/* Symmetric image<->spot contrastive loss, forward and backward in one call.
 *   MCLST_T_EYE       model.py:242-247: logits = S I^T / T; identity targets;
 *                     loss = (CE(logits, eye) + CE(logits^T, eye)) / 2
 *   MCLST_T_SOFT_DIV  baselines/Bleep/models.py:34-43: targets = softmax((I I^T + S S^T)/2/T),
 *   MCLST_T_SOFT_MUL  baselines/Bleep/models.py:70-79: ... /2*T; targets stay in the graph.
 * spot_emb, image_emb: [batch, dim] float32.  loss_out: one float32 (device).  d_spot /
 * d_image (both or neither): gradients of the loss w.r.t. the two inputs.  No batch x batch
 * matrix is held beyond one row block (scratch budget MCLST_LOSS_SCRATCH_MB, default 32768:
 * batches up to 32k rows then fit one block; smaller budgets stream row blocks).  The workspace
 * query takes the number of rows this call owns (= batch here). */
int mclst_contrastive_loss_workspace_bytes(int batch, int dim, int target_mode, int64_t rows_local,
                                           size_t* bytes);
int mclst_contrastive_loss(const float* spot_emb, int64_t ld_s, const float* image_emb, int64_t ld_i,
                           int batch, int dim, float temperature, int target_mode, float* loss_out,
                           float* d_spot, int64_t ld_ds, float* d_image, int64_t ld_di,
                           void* workspace, size_t workspace_bytes, mclst_stream_t stream);

/* ---------------------------------------------------------------- spot encoder pieces --- */

/* model.py:230-235: out[b,:] = expression[b,:] + x_table[long(position[b,0]),:]
 *                                              + y_table[long(position[b,1]),:]
 * (.long() truncation).  *error_flag (device uint32) is OR-ed with 1 when an index falls
 * outside [0, table_rows) -- nn.Embedding raises there; the caller checks it. */
int mclst_embed_add(const float* expression, int64_t ld_e, const float* position, int64_t ld_p,
                    const float* x_table, const float* y_table, int table_rows, int batch, int genes,
                    float* out, int64_t ld_o, uint32_t* error_flag, mclst_stream_t stream);
/* Backward of the gathers: DENSE [table_rows, genes] gradients (zero-filled, then
 * scatter-added), the layout torch.optim.Adam(weight_decay) of train.py:118-120 expects. */
int mclst_embed_add_backward(const float* d_out, int64_t ld_d, const float* position, int64_t ld_p,
                             int table_rows, int batch, int genes, float* d_x_table,
                             float* d_y_table, mclst_stream_t stream);
/* Same scatter-add WITHOUT the zero fill: the rows are added into whatever d_x_table / d_y_table
 * hold (gradient accumulation; or buffers the caller zero-filled earlier, off the critical path --
 * the fill of two [65536, genes] tables is 0.5 GB of writes that depend on nothing). */
/* x[0..n) = 0 by a grid of only `ctas` blocks: a fill that runs in the background of other work on
 * another stream instead of occupying every SM (x 16-byte aligned). */
int mclst_zero_fill_background(float* x, int64_t n, int ctas, mclst_stream_t stream);
int mclst_embed_add_backward_accumulate(const float* d_out, int64_t ld_d, const float* position,
                                        int64_t ld_p, int table_rows, int batch, int genes,
                                        float* d_x_table, float* d_y_table, mclst_stream_t stream);

/* nn.LayerNorm over the last dimension (model.py:13, :159): biased variance, eps inside the
 * square root; mean / rstd [rows] are kept for the backward. */
int mclst_layernorm_forward(const float* x, int64_t ld_x, const float* gamma, const float* beta,
                            int64_t rows, int cols, float eps, float* y, int64_t ld_y, float* mean,
                            float* rstd, mclst_stream_t stream);
int mclst_layernorm_backward(const float* dy, int64_t ld_dy, const float* x, int64_t ld_x,
                             const float* gamma, const float* mean, const float* rstd, int64_t rows,
                             int cols, float* dx, int64_t ld_dx, float* dgamma, float* dbeta,
                             float* scratch, size_t scratch_floats, mclst_stream_t stream);

/* nn.GELU() (exact erf form, model.py:25, :155) on n contiguous elements. */
int mclst_gelu_forward(const float* x, float* y, int64_t n, mclst_stream_t stream);
int mclst_gelu_backward(const float* dy, const float* x, float* dx, int64_t n, mclst_stream_t stream);

/* nn.Softmax(dim=-1) of model.py:41/:54 over `rows` rows of `cols` scores, in place; backward
 * overwrites d_probs with d_scores = probs * (d_probs - sum(d_probs * probs)). */
int mclst_softmax_forward(float* scores, int64_t ld, int64_t rows, int cols, mclst_stream_t stream);
int mclst_softmax_backward(const float* probs, float* d_probs_to_d_scores, int64_t ld, int64_t rows,
                           int cols, mclst_stream_t stream);

/* Block-diagonal softmax for the eval bank build (evel_her2st.py:24, 47-69: spots are embedded in
 * consecutive batches of `group`; attention never crosses a batch).  scores [rows, cols] holds
 * tiles of `cols` consecutive tokens (cols % group == 0); inside a token's own group the softmax
 * runs over the valid tokens (< n_valid), every other column becomes 0.  In place. */
int mclst_softmax_blockdiag(float* scores, int64_t ld, int64_t rows, int cols, int group,
                            int64_t n_valid, mclst_stream_t stream);

/* out[c] = sum_r x[r,c] (bias gradients), deterministic order. */
int mclst_col_sum(const float* x, int64_t ld, int64_t rows, int cols, float* out, mclst_stream_t stream);

/* ---------------------------------------------------------------- dense contractions ---- */

/* C_z[M,N] = act(alpha * op(A_z)[M,K] * op(B_z)[N,K]^T + bias[N]) + residual_z[M,N], z < batch
 * (row-major float32).  The building block behind every nn.Linear / einsum of the path and
 * their backward passes (model.py:25-27, :43-47, :51-57, :155-157).  a_trans = 0: A is stored
 * [M,K]; a_trans = 1: A is stored [K,M]; likewise B ([N,K] or [K,N]).  *_batch_stride are in
 * elements.  fp32 operands are split into fp16 hi/lo tiles and multiplied on the tensor cores
 * in three passes (precise = 1, ~fp32 accuracy) or one (precise = 0).  bias / residual may be
 * null (residual shares C's ld and batch stride); act: 0 none, 1 exact-erf GELU. */
int mclst_matmul_workspace_bytes(int64_t M, int64_t N, int64_t K, int batch, size_t* bytes);
int mclst_matmul(const float* A, int64_t lda, int a_trans, int64_t a_batch_stride,
                 const float* B, int64_t ldb, int b_trans, int64_t b_batch_stride,
                 float* C, int64_t ldc, int64_t c_batch_stride,
                 int64_t M, int64_t N, int64_t K, int batch, float alpha,
                 const float* bias, int act, const float* residual, int precise,
                 void* workspace, size_t workspace_bytes, mclst_stream_t stream);

/* ---------------------------------------------------------------- embedding-table Adam --- */

/* torch.optim.Adam(lr, betas, eps, weight_decay) as train.py:118-120 applies it to the position
 * tables x_embed / y_embed (model.py:204-205), without streaming 2 x 65536 x G parameters and
 * their moments through HBM on every step: rows a step does not touch are deferred and replayed
 * in registers (same arithmetic, step by step) when they are next read.  Lazy == dense bit for
 * bit; dense == torch up to fp32 rounding.
 *   coef_table   device buffer of mclst_adam_coef_bytes(max_steps) bytes: per-step scalars
 *   set_step     records the scalars of step `step` (1-based) -- call once per optimiser step
 *   dense        one step on n contiguous elements (grad nullable = zero data gradient)
 *   lazy_rows    for the distinct rows long(position[:, column]) of a batch: replay steps
 *                last_step[row]+1 .. steps_done; with d_out ([batch, genes], the gradient of the
 *                embed-add output) also apply step steps_done + 1 with the row's summed gradient.
 *                first_scratch: table_rows ints.  error_flag (device) is OR-ed with 1 when a
 *                position is outside [0, table_rows).  steps_done_dev (nullable, device int):
 *                when given it overrides steps_done at EXECUTION time, so that a launch captured
 *                in a CUDA graph follows the counter as training advances.
 *   lazy_flush   every row to steps_done (before state_dict / evaluation reads the table) */
size_t mclst_adam_coef_bytes(int max_steps);
int mclst_adam_set_step(void* coef_table, int max_steps, int step, double lr, double beta1,
                        double beta2, double eps, double weight_decay, mclst_stream_t stream);
int mclst_adam_dense(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                     const void* coef_table, int step, mclst_stream_t stream);
int mclst_adam_lazy_rows(float* table, float* exp_avg, float* exp_avg_sq, int* last_step,
                         int* first_scratch, int table_rows, int genes, const float* position,
                         int64_t ld_p, int column, int batch, const float* d_out, int64_t ld_d,
                         const void* coef_table, int steps_done, const int* steps_done_dev,
                         uint32_t* error_flag, mclst_stream_t stream);
int mclst_adam_lazy_flush(float* table, float* exp_avg, float* exp_avg_sq, int* last_step,
                          int table_rows, int genes, const void* coef_table, int steps_done,
                          mclst_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* MCLST_B200_H */
