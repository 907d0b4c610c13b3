/* credgcn.h -- C ABI of libcredgcn.so, the sm_100a implementation of the credibility-aware
 * LightGCN hot path (graph build -> K-layer propagation fwd/bwd -> BPR step with
 * popularity-aware negatives -> full-rank top-K evaluation).
 *
 * The reference (/root/reference, pure Python) has no FFI of its own: its de-facto boundary is
 * "Python names in a script + torch.sparse.mm" (SURVEY.md section 8b).  Each entry point below names
 * the reference code it replaces (file:line, CU = lightgcn_cu.py, V2 = Version-2/lighgcn_cu_pop.py,
 * DA = version_1/lightgcn_cu_pop_Degree-Aware Message.py).
 *
 * Conventions
 *   - every function returns 0 on success, a negative cgx_status on failure; the message is
 *     available from cgx_last_error() (thread-local);
 *   - every pointer marked "device" is a CUDA device pointer owned by the caller; the library
 *     never frees caller memory and keeps no global mutable state besides the tuning options of
 *     cgx_set_option (re-entrant per stream); it reads no environment variables;
 *   - scratch space is caller-provided: ask the matching *_workspace_bytes() first;
 *   - every op is asynchronous on the cudaStream_t passed as `stream` (a void* here so that the
 *     header needs no CUDA include); there are no hidden synchronisations except where a
 *     function documents a host-side result;
 *   - a NULL device pointer where one is required is CGX_ERR_ARG; there is no CPU fallback.
 *
 * Operator naming (the reference swaps M_ui / M_iu between CU and V2, so neither name is used):
 *     A : [U x I] user-row operator, base weight            (CU `M_iu`, V2 `M_ui`)
 *     C : [I x U] item-row operator, credibility weighted   (CU `M_ui`, V2 `M_iu`)
 */
#ifndef CREDGCN_H_
#define CREDGCN_H_

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#pragma GCC visibility push(default)   /* the library is built with -fvisibility=hidden */
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  CGX_OK = 0,
  CGX_ERR_ARG = -1,        /* bad argument (NULL pointer, unsupported emb_dim, size overflow) */
  CGX_ERR_WORKSPACE = -2,  /* workspace too small */
  CGX_ERR_CUDA = -3,       /* a CUDA runtime call or launch failed */
  CGX_ERR_UNSUPPORTED = -4
} cgx_status;

typedef enum { CGX_VARIANT_CU = 0, CGX_VARIANT_V2 = 1, CGX_VARIANT_DA = 2 } cgx_variant;
typedef enum { CGX_ORDER_JACOBI = 0, CGX_ORDER_GS = 1 } cgx_order;
typedef enum { CGX_SCORE_FP32 = 0, CGX_SCORE_BF16X3 = 1, CGX_SCORE_BF16 = 2 } cgx_score_precision;

const char* cgx_last_error(void);
int cgx_version(void);
/* Number of CUDA kernels this library has launched in this process (diagnostic tally). */
uint64_t cgx_launch_count(void);
/* Supported embedding widths: 16, 32, 64, 128, 256 (reference default emb_dim = 64, CU:53). */
int cgx_emb_dim_supported(int32_t d);

/* Process-wide tuning options (defaults in brackets).  None of them changes a result bit (tests force both sides),
 * the diagnostic bits 1-4 of CGX_OPT_EVAL_DEBUG excepted.
 * cgx_set_option stores `value` (negative = restore the default) and returns the previous one through
 * `previous` (nullable); cgx_get_option returns -1 for an unknown option. */
typedef enum {
  CGX_OPT_L2_TABLE_BYTES = 0,        /* [96 MiB] gathered tables above this are treated as HBM-resident by cgx_spmm */
  CGX_OPT_SPARSE_FIRST_ADJOINT = 1,  /* [1] cgx_propagate_bwd skips the zero rows of the loss gradient */
  CGX_OPT_PDL = 2,                   /* [1] programmatic dependent launch between consecutive SpMMs */
  CGX_OPT_P2P_ONESHOT_MAX = 3,       /* [2] cgx_comm_allreduce uses the one-shot form up to this many ranks */
  CGX_OPT_P2P_TIMING = 4,            /* [0] accumulate in-kernel phase times for cgx_comm_timing */
  CGX_OPT_P2P_TIMEOUT_MS = 5,        /* [20000] a cross-GPU barrier that waits longer gives up (cgx_comm_status) */
  CGX_OPT_EVAL_DEBUG = 6,            /* [0] diagnostics of cgx_eval_topk.  bit 0: print the redo-row count (synchronises);
                                        bits 1-4 switch parts of the tensor-core kernel off for timing (no list
                                        insertions / no MMAs / no TMA loads / no merges): WRONG RESULTS, profiles/eval_ablate.py */
  CGX_OPT_HOT_ROWS = 7,              /* [1] cgx_spmm uses the hot-row hints of cgx_csr.idx_hint when present */
  CGX_OPT_EVAL_GROUPS = 8,           /* [0] scanning warp groups of the tensor-core cgx_eval_topk: 0 = library choice, 1, 2 */
  CGX_OPT_TOPK_CHUNK_USERS = 9,      /* [0] users per chunk of cgx_eval_topk for k > 128: 0 = library choice (as many as
                                        its bounded workspace holds); a smaller value forces more, smaller chunks */
  CGX_OPT_COUNT_ = 10
} cgx_option;
int cgx_set_option(int option, int64_t value, int64_t* previous);
int64_t cgx_get_option(int option);

/* ------------------------------------------------------------------------------------------
 * Graph build.  Replaces edges_to_user_csr (CU:259-276), build_cred_weighted_mats (CU:368-399),
 * build_message_passing_mats (V2:429-452, DA:349-403): degree vectors, the user-row CSR used by
 * samplers/evaluators (neighbours ascending, duplicates kept) and both coalesced operators in
 * both orders.  Results are bit-exact against the reference's NumPy float32 arithmetic.
 * ------------------------------------------------------------------------------------------ */

/* One coalesced sparsity pattern in one row order with two value arrays.
 *   by user rows (n_rows = U): val_fwd = A values, val_bwd = C^T values
 *   by item rows (n_rows = I): val_fwd = C values, val_bwd = A^T values
 * perm / chunk_* are the SpMM work schedule (cgx_row_schedule): rows in descending degree order;
 * the first n_long of them exceed CGX_LONG_ROW non-zeros and are cut into CGX_CHUNK-sized chunks. */
typedef struct {
  int32_t n_rows;
  int32_t n_cols;
  int64_t nnz;
  const int64_t* indptr;     /* device, [n_rows + 1] */
  const int32_t* idx;        /* device, [nnz] column ids, ascending inside a row */
  const float* val_fwd;      /* device, [nnz] */
  const float* val_bwd;      /* device, [nnz] */
  const int32_t* perm;       /* device, [n_rows] row ids, descending degree (ties: ascending id) */
  int32_t n_long;            /* rows longer than CGX_LONG_ROW = perm[0 .. n_long) */
  int32_t n_chunks;          /* total chunks over all long rows */
  const int32_t* chunk_ptr;  /* device, [n_long + 1] first chunk of each long row (perm order) */
  const int32_t* chunk_row;  /* device, [n_chunks] position in perm of the row a chunk belongs to */
  int32_t n_huge;            /* rows longer than CGX_HUGE_ROW = perm[0 .. n_huge): combined by a finishing
                                kernel; the other long rows are combined by their last-arriving chunk */
  int32_t reserved_;
  int32_t* arrive;           /* device, [n_long] arrival counters, zero between launches (self-resetting);
                                mutable: at most one SpMM per cgx_csr may be in flight at a time */
  const void* work;          /* device, [n_chunks + n_rows - n_long] 16-byte work items in launch order
                                {int64 begin; int32 len; int32 row (or perm position of a chunk's row)} */
  const int32_t* idx_hint;   /* device, [nnz] or NULL: idx with bit 31 set where the column is a HOT row of the
                                gathered table (cgx_hot_hints); used by cgx_spmm when that table exceeds L2 */
} cgx_csr;

#define CGX_LONG_ROW 256     /* rows above this many non-zeros are split */
#define CGX_CHUNK 256        /* non-zeros per chunk of a split row */
#define CGX_HUGE_ROW 16384   /* rows above this (64 chunks) use the separate finishing kernel */

size_t cgx_graph_build_workspace_bytes(int64_t num_edges, int32_t num_users, int32_t num_items);

/* edges_u / edges_i: device int32[E] (the reference's on-disk int32 [2, E], CU:211).
 * cred: device float32[U] already clipped to [0, 1] (CU:359).
 * alpha: device float32[I], required for CGX_VARIANT_DA only: 1/log1p(max(deg_i,1)) computed with
 *        the caller's NumPy (libdevice log1pf is not bit-identical to NumPy's; DA:379-380).
 * deg_i_weights: NULL, or device int32[I] item degrees to use in the weight formulas instead of the
 *        histogram of these edges -- for a user-sharded build, where `edges` holds one shard's users
 *        but an item's degree counts its edges on every shard.
 * Outputs (all device, caller-allocated):
 *   deg_u int32[U], deg_i int32[I]                      np.bincount, duplicates counted
 *   samp_indptr int64[U+1], samp_idx int32[E]           edges_to_user_csr
 *   by_user:  indptr int64[U+1], idx int32[E], val_fwd/val_bwd float32[E]   (first nnz entries valid)
 *   by_item:  indptr int64[I+1], idx int32[E], val_fwd/val_bwd float32[E]
 *   nnz_out  int64[2]                                   [0] coalesced non-zero count (<= E),
 *                                                       [1] number of out-of-range edges (must be 0)
 * deg_only != 0 stops after the degree vectors (used to compute `alpha` for the DA variant). */
int cgx_graph_build(const int32_t* edges_u, const int32_t* edges_i, int64_t num_edges,
                    int32_t num_users, int32_t num_items, const float* cred, int variant,
                    const float* alpha, const int32_t* deg_i_weights, int32_t* deg_u, int32_t* deg_i,
                    int64_t* samp_indptr, int32_t* samp_idx,
                    int64_t* user_indptr, int32_t* user_idx, float* user_val_fwd, float* user_val_bwd,
                    int64_t* item_indptr, int32_t* item_idx, float* item_val_fwd, float* item_val_bwd,
                    int64_t* nnz_out, int deg_only, void* workspace, size_t workspace_bytes, void* stream);

/* Only the user-row CSR of an edge list (val/test splits): edges_to_user_csr, CU:259-276. */
int cgx_user_csr(const int32_t* edges_u, const int32_t* edges_i, int64_t num_edges, int32_t num_users,
                 int32_t num_items, int64_t* indptr, int32_t* idx, void* workspace,
                 size_t workspace_bytes, void* stream);

/* SpMM work schedule of one row order.  cgx_row_schedule sorts rows by descending degree into
 * perm int32[n_rows] and returns (host results; synchronises `stream`) how many rows exceed
 * CGX_LONG_ROW and how many chunks they make; cgx_row_schedule_chunks then fills
 * chunk_ptr int32[n_long+1] / chunk_row int32[n_chunks] -- call it with the SAME workspace, untouched
 * in between, and only when n_long > 0. */
size_t cgx_row_schedule_workspace_bytes(int32_t n_rows);
int cgx_row_schedule(const int64_t* indptr, int32_t n_rows, int32_t* perm, int32_t* n_long_host,
                     int32_t* n_chunks_host, int32_t* n_huge_host, void* workspace, size_t workspace_bytes,
                     void* stream);
int cgx_row_schedule_chunks(int32_t n_rows, int32_t n_long, int32_t n_chunks, int32_t* chunk_ptr,
                            int32_t* chunk_row, void* workspace, size_t workspace_bytes, void* stream);
/* Flattens the schedule into the 16-byte work items the SpMM kernel streams (one load per item instead
 * of the perm -> indptr -> chunk table pointer chase): work = device buffer of
 * 16 * (n_chunks + n_rows - n_long) bytes.  chunk_ptr / chunk_row may be NULL when n_long == 0. */
int cgx_row_schedule_work(const int64_t* indptr, const int32_t* perm, int32_t n_rows, int32_t n_long,
                          int32_t n_chunks, const int32_t* chunk_ptr, const int32_t* chunk_row, void* work,
                          void* stream);

/* Hot-row hints of one row order (north_star: "staging of hot (high-degree) rows").  When the gathered table is
 * larger than the L2 cache, cgx_spmm loads the rows of the n_hot highest-degree COLUMNS with the L2 evict_last
 * priority and streams everything else (cold rows, ids / values, running sums, outputs) through evict_first, so
 * that the rows most edges point at stay resident.  col_by_degree = the other row order's `perm` (columns in
 * descending degree); n_hot is normally hot_bytes / (4 * emb_dim).  idx_hint int32[nnz] = idx | hot << 31.
 * The hints change no result bit. */
size_t cgx_hot_hints_workspace_bytes(int32_t n_cols);
int cgx_hot_hints(const int32_t* idx, int64_t nnz, int32_t n_cols, const int32_t* col_by_degree, int32_t n_hot,
                  int32_t* idx_hint, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Propagation.  Replaces torch.sparse.mm + stack().mean() (CU:420-448, V2:472-490) and their
 * autograd (CU:651, V2:862).  fp32, <= 1e-4 relative to the reference.
 * ------------------------------------------------------------------------------------------ */

/* One CSR SpMM with the fused epilogue, per output row r (y = sum_j val[j] * X[idx[j], :]):
 *     if Y:       Y[r]       = y
 *     if ACC_OUT: ACC_OUT[r] = acc_scale * (ACC_IN[r] + y)      (ACC_IN may be NULL -> 0; may alias ACC_OUT)
 * The forward uses ACC for the running layer sum (last layer: acc_scale = 1/(K+1)); the backward
 * uses it for "gradient seed + transposed product".  use_bwd_values selects val_bwd.
 * workspace: cgx_spmm_workspace_bytes() (partials of the long-row chunks). */
size_t cgx_spmm_workspace_bytes(const cgx_csr* m, int32_t d);
int cgx_spmm(const cgx_csr* m, int use_bwd_values, int32_t d, const float* X, float* Y,
             const float* ACC_IN, float* ACC_OUT, float acc_scale,
             void* workspace, size_t workspace_bytes, void* stream);

/* The same product when most rows of X are zero (the loss gradient touches <= 3 * batch rows, so the first
 * adjoint product of loss.backward() -- CU:651, V2:862 -- gathers mostly zeros): x_row_nonzero[c] == 0
 * promises that row c of X is all zero, and such rows are not loaded.  Same result as cgx_spmm.
 * cgx_row_flags writes the flags for a table (1 = the row has a non-zero entry; -0.0 counts as zero). */
int cgx_spmm_sparse_rows(const cgx_csr* m, int use_bwd_values, int32_t d, const float* X,
                         const uint8_t* x_row_nonzero, float* Y, const float* ACC_IN, float* ACC_OUT,
                         float acc_scale, void* workspace, size_t workspace_bytes, void* stream);
int cgx_row_flags(const float* X, int64_t n_rows, int32_t d, uint8_t* flags, void* stream);
/* The general form: both flag arrays are optional.  acc_row_nonzero[r] == 0 promises that row r of ACC_IN is all
 * zero, and it is then not read (the adjoint adds the row-sparse loss gradient to every layer). */
int cgx_spmm_ex(const cgx_csr* m, int use_bwd_values, int32_t d, const float* X, const uint8_t* x_row_nonzero,
                float* Y, const float* ACC_IN, const uint8_t* acc_row_nonzero, float* ACC_OUT, float acc_scale,
                void* workspace, size_t workspace_bytes, void* stream);

/* cgx_spmm picks its thread geometry by regime: a gathered table X of more than this many bytes is treated as
 * HBM-resident (narrower groups, more rows in flight), a smaller one as L2-resident.  Default 96 MiB; a negative
 * value restores the default.  Returns the previous value.  Results do not depend on it (tests force both).
 * Same as cgx_set_option(CGX_OPT_L2_TABLE_BYTES, ...). */
int64_t cgx_spmm_set_l2_table_bytes(int64_t bytes);

size_t cgx_propagate_workspace_bytes(const cgx_csr* by_user, const cgx_csr* by_item, int32_t d);
/* The same for one layer order: Gauss-Seidel needs one layer buffer per side, Jacobi two (the size above). */
size_t cgx_propagate_workspace_bytes_for(const cgx_csr* by_user, const cgx_csr* by_item, int32_t d, int order);

/* Forward: final = mean over layers 0..K.  order JACOBI = CU:429-437, GS = V2:482-486.
 * e0_u [U,d], e0_i [I,d] -> out_u [U,d], out_i [I,d].  Nothing is saved for backward (the
 * operators are constants, so the adjoint needs only the output gradients). */
int cgx_propagate_fwd(const cgx_csr* by_user, const cgx_csr* by_item, int order, int32_t num_layers,
                      int32_t d, const float* e0_u, const float* e0_i, float* out_u, float* out_i,
                      void* workspace, size_t workspace_bytes, void* stream);
/* The same forward, layers [layer_begin, layer_end) only (0 <= layer_begin <= layer_end <= num_layers), with
 * output-row masks for the last layer's products.  A call that starts at layer k > 0 continues the one that ran
 * layers 0..k-1 on the same out_u / out_i and workspace.  rows_u uint8[U] / rows_i uint8[I] (nullable): the last
 * layer computes and writes (out_* and its layer buffer) only the flagged rows; the other rows of out_* keep the
 * running sum of layers 0..K-1.  Masked rows can be computed later by a call for layer K-1 alone with the
 * complementary masks on the same workspace: the last layer's inputs are not overwritten by it, and the final
 * tables then carry the bits of cgx_propagate_fwd.  all_rows: uint8[max(U, I)], every entry 1, needed with a mask.
 * (The last layer adds into out_* in place: computing a row twice adds it twice.)  The completing call picks its
 * SpMM geometry from the options current when it runs (CGX_OPT_L2_TABLE_BYTES): change none between the two calls,
 * or the completed rows may differ from cgx_propagate_fwd in the last bits. */
int cgx_propagate_fwd_layers(const cgx_csr* by_user, const cgx_csr* by_item, int order, int32_t num_layers,
                             int32_t d, const float* e0_u, const float* e0_i, float* out_u, float* out_i,
                             int32_t layer_begin, int32_t layer_end, const uint8_t* rows_u, const uint8_t* rows_i,
                             const uint8_t* all_rows, void* workspace, size_t workspace_bytes, void* stream);

/* Backward: (g_u, g_i) = dL/d(out_u, out_i) dense -> (d_e0_u, d_e0_i).  SURVEY.md appendix C. */
int cgx_propagate_bwd(const cgx_csr* by_user, const cgx_csr* by_item, int order, int32_t num_layers,
                      int32_t d, const float* g_u, const float* g_i, float* d_e0_u, float* d_e0_i,
                      void* workspace, size_t workspace_bytes, void* stream);
/* The same when the caller already knows which rows of g_u / g_i are non-zero (uint8 flags as cgx_row_flags writes
 * them; every unflagged row MUST be all zero): saves the scan of both tables.  cgx_bpr_mark_rows provides the flags
 * for the gradient of cgx_bpr_fwd_bwd.  Pass both arrays or neither (NULL, NULL = cgx_propagate_bwd). */
int cgx_propagate_bwd_flagged(const cgx_csr* by_user, const cgx_csr* by_item, int order, int32_t num_layers,
                              int32_t d, const float* g_u, const float* g_i, const uint8_t* g_u_rows,
                              const uint8_t* g_i_rows, float* d_e0_u, float* d_e0_i, void* workspace,
                              size_t workspace_bytes, void* stream);
/* The same backward of loss.backward() (CU:651, V2:862), told where the first item-side adjoint can be non-zero.
 * front_i uint8[I] (nullable; NULL = cgx_propagate_bwd_flagged): every item row that is non-zero in g_i, or that
 * has a non-zero row of g_u among its neighbours, MUST be flagged -- cgx_batch_frontier writes such flags for the
 * gradient of a triple batch.  The first item-row product g_i + A^T g_u then computes only the flagged rows when
 * its output is scratch (Gauss-Seidel always, Jacobi for num_layers >= 2), and the product that reads it gathers
 * only those rows.  Same bits as cgx_propagate_bwd_flagged. */
int cgx_propagate_bwd_frontier(const cgx_csr* by_user, const cgx_csr* by_item, int order, int32_t num_layers,
                               int32_t d, const float* g_u, const float* g_i, const uint8_t* g_u_rows,
                               const uint8_t* g_i_rows, const uint8_t* front_i, float* d_e0_u, float* d_e0_i,
                               void* workspace, size_t workspace_bytes, void* stream);
/* Item frontier of a triple batch for cgx_propagate_bwd_frontier (the items whose rows the first adjoint of
 * loss.backward(), CU:651 / V2:862, can make non-zero): flags_i uint8[num_items] is zeroed, then set for pos[t],
 * neg[t] and every column of by_user row users[t], t < batch.  users / pos / neg int64[batch] (device); ids out of
 * range count as 0, as in cgx_bpr_plan.  flags_u uint8[num_users] (nullable) is zeroed and set for users[t]: the
 * user rows the loss reads.  Depends on the indices only: it can run on a side stream beside the forward
 * propagation, as cgx_bpr_plan does. */
int cgx_batch_frontier(const cgx_csr* by_user, const int64_t* users, const int64_t* pos, const int64_t* neg,
                       int64_t batch, uint8_t* flags_i, uint8_t* flags_u, void* stream);

/* ------------------------------------------------------------------------------------------
 * BPR + L2 (+ fairness) on a batch of (user, pos, neg) triples.  Replaces score / l2_reg / the loss
 * assembly (CU:450-463, 635-648) and bpr_loss (V2:495-508) with their backward.
 *   L = -mean(log(sigmoid(y+ - y-) + 1e-12)) + fair * mean(pop[pos] * y+)
 *       + reg * mean(|e0_u[u]|^2 + |e0_i[p]|^2 + |e0_i[n]|^2)
 * Gradients are scattered without atomics: the 3B (row, triple) pairs are sorted (cgx_bpr_plan) and
 * each distinct row is summed by one thread group in triple order (deterministic).
 *   g_u [U,d], g_i [I,d]   dL/d(propagated tables); must be zero-filled by the caller; only the
 *                          rows named by the batch are written
 *   ego_rows int32[3B], ego_coef float[3B]   compact L2 gradient: after the backward propagation
 *                          add ego_coef[k] * e0[row] to d_e0 at row = ego_rows[k] for every k with
 *                          ego_rows[k] >= 0 (rows >= U are items, offset by U; each row appears once)
 *                          -- done by cgx_bpr_apply_ego
 *   loss_out float[1]      NaN if any index of the batch was out of range
 *   batch_total            the mean's denominator: `batch`, or -- when the batch is sharded over ranks -- the
 *                          global batch size (the rank losses then add up to the global loss)
 * ------------------------------------------------------------------------------------------ */
/* Scatter plan: the 3B (row, entry) keys of a batch sorted by row, uint64[3B] (device).  Depends on
 * the indices only -- build it on a side stream while the forward propagation runs. */
size_t cgx_bpr_plan_workspace_bytes(int64_t batch);
int cgx_bpr_plan(const int64_t* users, const int64_t* pos, const int64_t* neg, int64_t batch,
                 int32_t num_users, int32_t num_items, uint64_t* plan,
                 void* workspace, size_t workspace_bytes, void* stream);
size_t cgx_bpr_workspace_bytes(int64_t batch, int32_t num_users, int32_t num_items);
int cgx_bpr_fwd_bwd(const int64_t* users, const int64_t* pos, const int64_t* neg, int64_t batch,
                    int64_t batch_total, const uint64_t* plan, int32_t num_users, int32_t num_items, int32_t d,
                    const float* f_u, const float* f_i, const float* e0_u, const float* e0_i,
                    const float* pop, float reg_weight, float fair_weight,
                    float* loss_out, float* g_u, float* g_i,
                    int32_t* ego_rows, float* ego_coef,
                    void* workspace, size_t workspace_bytes, void* stream);
int cgx_bpr_apply_ego(const int32_t* ego_rows, const float* ego_coef, int64_t n_entries,
                      int32_t num_users, int32_t d, const float* e0_u, const float* e0_i,
                      float* d_e0_u, float* d_e0_i, void* stream);
/* Row bookkeeping for callers that keep g_u / g_i all-zero between steps instead of zero-filling (U + I) d floats
 * per step: ego_rows (output of cgx_bpr_fwd_bwd) names every distinct row the batch wrote.
 *   cgx_bpr_mark_rows   nz_u[row] = 1 / nz_i[row] = 1 for those rows (flags for cgx_propagate_bwd_flagged;
 *                       uint8[U] / uint8[I], zero before the first step)
 *   cgx_bpr_clear_rows  zeroes those rows of g_u / g_i and their flags again (call after the backward) */
int cgx_bpr_mark_rows(const int32_t* ego_rows, int64_t n_entries, int32_t num_users, uint8_t* nz_u, uint8_t* nz_i,
                      void* stream);
int cgx_bpr_clear_rows(const int32_t* ego_rows, int64_t n_entries, int32_t num_users, int32_t d, float* g_u,
                       float* g_i, uint8_t* nz_u, uint8_t* nz_i, void* stream);

/* ------------------------------------------------------------------------------------------
 * Samplers.  Replace sample_pos_item / sample_neg_item (CU:288-299) and
 * sample_neg_item_popmix with its popularity law (V2:349-376, 805-810).  Counter-based Philox4x32-10:
 * the triple of batch slot k under (seed, offset) never depends on launch geometry.
 * The popularity law p_i ~ (deg_i + 1)^gamma is held as an alias table over DEGREE CLASSES (all
 * items of equal degree share one class) plus the item list ordered by degree -- the same
 * distribution as an alias table over items, with a table small enough to stay cache resident.
 * ------------------------------------------------------------------------------------------ */
size_t cgx_sampler_build_workspace_bytes(int32_t num_items);
/* Outputs (device): items_by_deg int32[I]; class_start int32[I+1], class_prob float[I],
 * class_alias int32[I] (first n_classes entries valid); n_classes int32[1]. */
int cgx_sampler_build(const int32_t* deg_i, int32_t num_items, double gamma,
                      int32_t* items_by_deg, int32_t* class_start, float* class_prob,
                      int32_t* class_alias, int32_t* n_classes,
                      void* workspace, size_t workspace_bytes, void* stream);

/* users int64[B]: batch users (each must own >= 1 train item, as CU:592 guarantees).
 * mix_pop < 0 selects the uniform sampler of CU:295-299 (tables may then be NULL).
 * After max_tries rejected proposals the kernel falls back to uniform proposals (V2:373-376).
 * offset_dev (nullable): device counter added to `offset`, so that a captured CUDA graph draws new
 * triples on every replay (advance it with cgx_tick). */
int cgx_sample_triples(const int64_t* users, int64_t batch, const int64_t* samp_indptr,
                       const int32_t* samp_idx, int32_t num_items,
                       const int32_t* items_by_deg, const int32_t* class_start,
                       const float* class_prob, const int32_t* class_alias, const int32_t* n_classes,
                       float mix_pop, int32_t max_tries, uint64_t seed, uint64_t offset,
                       const uint64_t* offset_dev, int64_t* pos_out, int64_t* neg_out, void* stream);

/* ------------------------------------------------------------------------------------------
 * Optimiser.  Replaces torch.optim.Adam(lr).step() (CU:587,652; V2:793,863; torch defaults) on the two
 * embedding tables in one launch.  step = step_host + *step_dev (step_dev nullable), 1-based.
 * cgx_tick increments a device counter by one (graph-replayable step / sampler offsets).
 * ------------------------------------------------------------------------------------------ */
int cgx_tick(uint64_t* counter, void* stream);
int cgx_adam_step(float* p0, const float* g0, float* m0, float* v0, int64_t n0,
                  float* p1, const float* g1, float* m1, float* v1, int64_t n1,
                  float lr, float beta1, float beta2, float eps,
                  const uint64_t* step_dev, int64_t step_host, void* stream);

/* ------------------------------------------------------------------------------------------
 * Multi-GPU item-table exchange over NVLink peer memory (user-sharded propagation, SURVEY.md section 8e; the
 * reference is single-device).  One communication buffer per rank: cgx_comm_alloc (cudaMalloc, zeroed),
 * cgx_comm_ipc_handle -> 64-byte cudaIpcMemHandle_t to hand to the peers, cgx_comm_ipc_open on their
 * side.  cgx_comm_allreduce sums n_floats float32 at byte offset in_off of every rank's buffer, in rank
 * order (deterministic), into byte offset out_off of every rank's buffer: a two-shot pull kernel with
 * system-scope flag barriers at flag_off (>= 4 * (2 * world + 2) bytes, zero before first use).
 * The barrier waits are bounded (CGX_OPT_P2P_TIMEOUT_MS): a rank that never arrives makes the waiting kernels
 * give up, record an error word in the flag page and finish (with an unusable result) instead of hanging every
 * GPU of the job; cgx_comm_status reads that word (synchronises the device; 0 = no time-out so far, else
 * (barrier << 8 | peer rank + 1) of the first wait that expired, barrier 1 = A, 2 = B).
 * peer_bases: host array of `world` device pointers (own buffer at index rank).  epoch_dev: device counter
 * holding 1, 2, 3, ... for successive exchanges (cgx_tick it before each call), the same on all ranks.
 * ------------------------------------------------------------------------------------------ */
int cgx_comm_alloc(size_t bytes, void** base_out);
int cgx_comm_free(void* base);
int cgx_comm_ipc_handle(void* base, void* handle_out_64);
int cgx_comm_ipc_open(const void* handle_64, void** peer_base_out);
int cgx_comm_ipc_close(void* peer_base);
int cgx_comm_allreduce(int rank, int world, void* const* peer_bases, size_t in_off, size_t out_off,
                       size_t flag_off, int64_t n_floats, const uint64_t* epoch_dev, void* stream);
int cgx_comm_status(const void* base, size_t flag_off, int world, uint32_t* error_out);
/* The same exchange through the NVSwitch (NVLS): the `world` buffers must be bound to one multicast object whose
 * mapping is mc_base (same offsets as the unicast mappings in peer_bases; e.g. torch symmetric memory).  Rank r sums
 * slice r inside the switch (multimem.ld_reduce) and the switch replicates the result into every rank's out region
 * (multimem.st): about half the NVLink traffic of the pull form.  Every rank receives identical bits; the order of
 * the in-switch sum is the switch's, so the last place may differ from cgx_comm_allreduce. */
int cgx_comm_allreduce_nvls(int rank, int world, void* const* peer_bases, void* mc_base, size_t in_off,
                            size_t out_off, size_t flag_off, int64_t n_floats, const uint64_t* epoch_dev, void* stream);
/* All-gather of one block of bytes_per_rank bytes (16-byte granularity) per rank: block `rank` is read from the
 * local device pointer src and lands at byte offset dst_off + rank * bytes_per_rank of EVERY rank's buffer; returns
 * when all `world` blocks are local.  One epoch tick like the all-reduces.  Used for the compact loss gradient of the
 * user-sharded step (<= 2 * batch item rows per rank instead of two dense item tables). */
int cgx_comm_allgather(int rank, int world, void* const* peer_bases, const void* src, size_t dst_off,
                       size_t flag_off, int64_t bytes_per_rank, const uint64_t* epoch_dev, void* stream);

/* Fused product + exchange of the user-sharded propagation.  cgx_spmm_push is cgx_spmm(Y only) whose output row r is
 * stored straight into the communication buffer of the rank that owns row r (rows_per consecutive rows per rank,
 * owner = r / rows_per), at stage_off + ((rank * rows_per + r % rows_per) * d) floats -- posted NVLink stores issued
 * from the SpMM epilogue while the rest of the product is still being gathered (x_row_nonzero: optional row flags,
 * as in cgx_spmm_sparse_rows).  cgx_spmm_set_push_peers registers the peer-mapped buffers once (index = rank).
 * cgx_comm_allreduce_pushed then sums, on every owner, the `world` staged copies of its rows with LOCAL loads (rank
 * order: the bits of cgx_comm_allreduce), stores the reduced rows into every rank's out region (float[n_rows, d] at
 * out_off) and returns when all rows of all owners have arrived.  Needs world * rows_per * d * 4 bytes at stage_off. */
int cgx_spmm_set_push_peers(void* const* peer_bases, int world);
int cgx_spmm_push(const cgx_csr* m, int use_bwd_values, int32_t d, const float* X, const uint8_t* x_row_nonzero,
                  size_t stage_off, int rank, int world, int32_t rows_per,
                  void* workspace, size_t workspace_bytes, void* stream);
int cgx_comm_allreduce_pushed(int rank, int world, void* const* peer_bases, size_t stage_off, size_t out_off,
                              size_t flag_off, int64_t n_rows, int32_t d, int32_t rows_per,
                              const uint64_t* epoch_dev, void* stream);

/* Diagnostics (CGX_OPT_P2P_TIMING = 1): nanoseconds accumulated inside cgx_comm_allreduce's kernel in
 * {barrier A, reduce + delivery, barrier B} and the number of exchanges since the last call; out4 is a HOST array.
 * Synchronises the device.  All zeros when timing is off. */
int cgx_comm_timing(uint64_t* out4);

/* ------------------------------------------------------------------------------------------
 * Full-rank evaluation.  Replaces the per-user loop of evaluate_full_ranking (V2:691-704):
 * scores of `users` against every item, train items forced to -1e9, best K by
 * (score desc, item id asc).  out_ids int32[n, K], out_scores float[n, K].
 * 0 < k <= min(4096, num_items); a larger k fails with CGX_ERR_ARG.
 *   k <= 128   CGX_SCORE_FP32: the exact fp32 kernel.  BF16X3 / BF16: the tcgen05 kernel where
 *              cgx_eval_topk_uses_tensor_cores says so (BF16X3 with the same ids and score bits as fp32, BF16 a
 *              single-pass selection re-scored in fp32), else the fp32 kernel.
 *   k > 128    every precision runs the exact fp32 deep kernel: ids and score bits equal those of FP32, and the
 *              first 128 columns equal a k = 128 FP32 call (CGX_SCORE_BF16 also gets the exact result).  The
 *              workspace is bounded (about 1 GiB); users are processed in chunks that fit it
 *              (CGX_OPT_TOPK_CHUNK_USERS).
 * ------------------------------------------------------------------------------------------ */
size_t cgx_eval_topk_workspace_bytes(int64_t n_users, int32_t num_items, int32_t d, int32_t k,
                                     int precision);
int cgx_eval_topk(const int64_t* users, int64_t n_users, const float* f_u, const float* f_i,
                  int32_t num_items, int32_t d, const int64_t* train_indptr, const int32_t* train_idx,
                  int32_t k, int precision, int32_t* out_ids, float* out_scores,
                  void* workspace, size_t workspace_bytes, void* stream);

/* 1 when cgx_eval_topk runs the tcgen05 kernel for this (d, k, precision); 0 when it falls back to an exact
 * fp32 kernel (precision FP32, k > 52, or a width whose operands do not fit shared memory: BF16X3 with d = 256). */
int cgx_eval_topk_uses_tensor_cores(int32_t d, int32_t k, int precision);

/* Scores of explicit candidate lists (sampled protocol, CU:521-527): cand int64[n, C] ->
 * scores float[n, C] = <f_u[users[r]], f_i[cand[r, c]]>. */
int cgx_score_candidates(const int64_t* users, const int64_t* cand, int64_t n_users, int32_t n_cand,
                         int32_t d, const float* f_u, const float* f_i, float* scores, void* stream);

/* Candidate lists of the sampled protocol drawn on device (CU:505-521): cand int64[n, 1 + n_neg]; column 0
 * is one of the user's test items (uniform), the others are uniform items outside test U train (rejection by
 * binary search in both sorted rows).  users must each own >= 1 test item.  Philox streams per (user, slot). */
int cgx_eval_candidates(const int64_t* users, int64_t n_users, const int64_t* train_indptr,
                        const int32_t* train_idx, const int64_t* test_indptr, const int32_t* test_idx,
                        int32_t num_items, int32_t n_neg, uint64_t seed, int64_t* cand, void* stream);

/* ranked[r] = cand[r] reordered by descending score, ties keeping candidate order (np.argsort(-scores),
 * CU:527, made stable). */
int cgx_rank_candidates(const float* scores, const int64_t* cand, int64_t n_users, int32_t n_cand,
                        int64_t* ranked, void* stream);

/* Ranking metrics from ranked ids int32[n, ld] (rows of cgx_eval_topk, or cgx_rank_candidates narrowed to
 * int32), accumulated in double like the reference's Python floats: metrics_at_k CU:469-484 / V2:514-530 and
 * the accumulation loops of evaluate_full_ranking V2:691-752 / evaluate_sampled CU:521-546.
 *   ground truth   gt_single != NULL: one item per row (sampled protocol), else the sorted test rows
 *                  test_idx[test_indptr[users[r]] .. test_indptr[users[r] + 1]) (duplicates counted, as np.diff)
 *   ks_host        HOST array of n_ks <= 8 ascending cut-offs, each <= min(ld, 4096)
 *   item_pop       nullable int64[num_items] train popularity (V2:382-388); total_train = its sum
 *   group          nullable uint8[n]: bit 0 = row is in the high-credibility group, bit 1 = in the low one
 *                  (make_cred_groups V2:406-423; a row can be in both when the groups overlap)
 *   bitmaps        nullable uint32[n_ks][ceil(num_items / 32)], ZEROED BY THE CALLER: bit i of bitmap ki is set
 *                  when item i occurs in columns [ks[ki-1], ks[ki]) of some row; a user-sharded evaluation ORs
 *                  the bitmaps of all ranks before cgx_eval_coverage
 *   out            device double[n_ks][7]: SUMS over rows of precision, recall, ndcg, mean_k log(pop + 1),
 *                  mean_k -log2((pop + 1) / (total_train + num_items)), recall of group 1, recall of group 2
 * Deterministic: block partials are combined in a fixed order. */
size_t cgx_eval_metrics_workspace_bytes(int64_t n_users, int32_t n_ks);
int cgx_eval_metrics(const int32_t* ranked, int64_t n_users, int32_t ld, const int64_t* users,
                     const int64_t* test_indptr, const int32_t* test_idx, const int32_t* gt_single,
                     int32_t num_items, const int32_t* ks_host, int32_t n_ks, const int64_t* item_pop,
                     int64_t total_train, const uint8_t* group, uint32_t* bitmaps, double* out,
                     void* workspace, size_t workspace_bytes, void* stream);

/* counts[ki] = distinct items in the first ks[ki] columns = popcount(bitmaps[0] | .. | bitmaps[ki])
 * (item_coverage numerator, V2:708-712).  counts: device uint64[n_ks], overwritten. */
int cgx_eval_coverage(const uint32_t* bitmaps, int32_t num_items, int32_t n_ks, uint64_t* counts, void* stream);

#ifdef __cplusplus
}
#endif
#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#endif /* CREDGCN_H_ */
