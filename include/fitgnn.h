/*
 * fitgnn.h — C ABI of libfitgnn_b200.so (sm_100a).
 *
 * The reference (Roy-Shubhajit/FIT-GNN) is pure Python and has no FFI; the seam this
 * library sits behind is the PyG operator/model surface the reference calls
 * (SURVEY.md §8b).  Every entry point names the reference call site it replaces.
 *
 * Conventions
 *   - every function returns 0 on success, a negative FITGNN_E* code otherwise and never
 *     throws/aborts across the ABI; fitgnn_last_error() returns the message of the last
 *     failure on the calling thread;
 *   - all data pointers are DEVICE pointers unless a parameter is named host_*;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream);
 *   - the library never allocates caller-visible memory: outputs and workspaces are
 *     caller-owned; data-dependent output sizes come from a *_plan call that leaves its
 *     intermediates in the workspace for the matching *_fill call;
 *   - a filled pack is immutable; calls are re-entrant for distinct (pack, ws, stream);
 *   - dense matrices are row-major fp32 with an explicit leading dimension in elements.
 */
#ifndef FITGNN_H_
#define FITGNN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FITGNN_ABI_VERSION 1

enum {
  FITGNN_OK = 0,
  FITGNN_EINVAL = -1,   /* bad argument (null pointer, negative size, unknown mode) */
  FITGNN_ECUDA = -2,    /* a CUDA runtime / driver call failed                        */
  FITGNN_ERANGE = -3,   /* sizes exceed what the int32 / packed-key layout can hold    */
  FITGNN_EWS = -4,      /* workspace too small                                         */
  FITGNN_EUNSUP = -5    /* shape not supported by the requested kernel                 */
};

/* activation fused into SpMM / GEMM epilogues (network.py:32 uses ELU, alpha = 1) */
enum { FITGNN_ACT_NONE = 0, FITGNN_ACT_ELU = 1 };

/* head applied after lt1 (network.py:35 log_softmax; :64 identity; :95,:135 softmax) */
enum { FITGNN_HEAD_IDENTITY = 0, FITGNN_HEAD_LOG_SOFTMAX = 1, FITGNN_HEAD_SOFTMAX = 2 };

/* subgraph augmentation (utils.py:190 cluster_node, :235 extra_node, else none) */
enum { FITGNN_MODE_NONE = 0, FITGNN_MODE_EXTRA = 1, FITGNN_MODE_CLUSTER = 2 };

/* segment pooling (network.py:93,131 global_max_pool; :164,202 global_mean_pool) */
enum { FITGNN_POOL_MAX = 0, FITGNN_POOL_MEAN = 1 };

/* GEMM arithmetic.  FP32 = exact fp32 FMA on CUDA cores; BF16X3 = tcgen05 tensor cores on
 * a hi/lo bf16 split of both operands (3 MMAs, ~2^-17 relative operand error). */
enum { FITGNN_GEMM_FP32 = 0, FITGNN_GEMM_BF16X3 = 1, FITGNN_GEMM_FP16X2 = 2 /* fitgnn_gemm_f16 & co. only */ };

/*
 * Packed block-diagonal CSR of all subgraphs Gs (replaces the list[Data] built by
 * coarsening_classification utils.py:186-267 and re-collated by G_DataLoader run.py:336).
 * Row r of the pack is one subgraph-local node; rows of one subgraph are contiguous and in
 * the reference's node order (M.orig_idx ascending, then cluster nodes in first-seen order).
 * CSR row = message target, col = message source, self loop included, duplicates kept
 * (PyG gcn_norm semantics, SURVEY §8a-a1).  Edge weight = dinv[row] * dinv[col].
 */
typedef struct fitgnn_pack {
  int64_t n_rows;           /* N' */
  int64_t nnz;              /* E' + N' */
  int64_t n_sub;            /* k */
  int64_t n_core;           /* number of core rows (= N for a node task) */
  int64_t n_src;            /* rows of the de-duplicated feature table gid points into */
  const int32_t* rowptr;    /* [n_rows+1] */
  const int32_t* col;       /* [nnz] pack-local source row, ascending inside a row */
  const float* dinv;        /* [n_rows] deg^-1/2, deg = row length (self loop counted) */
  const int32_t* gid;       /* [n_rows] global node id, or N + cluster id for a cluster node */
  const int32_t* sub_ptr;   /* [n_sub+1] first row of each subgraph */
  const int32_t* core_rows; /* [n_core] pack rows of core nodes, ascending */
  const uint8_t* is_core;   /* [n_rows] 1 = node belongs to the subgraph's own cluster */
  const uint8_t* mask;      /* [n_rows] M.mask exactly as the reference stores it (utils.py:260-265) */
} fitgnn_pack;

/* result of fitgnn_pack_plan: the data-dependent sizes the caller allocates the pack from, the size
 * of the second workspace fitgnn_pack_fill needs, and private state carried from plan to fill */
typedef struct fitgnn_plan {
  int64_t n_rows, nnz, n_sub, n_core, n_src;
  int64_t fill_ws_bytes;
  int64_t priv[27];
} fitgnn_plan;

int fitgnn_abi_version(void);
/* copies the calling thread's last error message (NUL terminated) into buf; returns its length */
int fitgnn_last_error(char* buf, size_t n);
/* SM count and compute capability (major*10+minor) of the current device */
int fitgnn_device_info(int* sm_count, int* cc);
/* Kernel-tuning switches (A/B measurements only; results never depend on them — except gemm_debug, which exists to BREAK
 * them for a measurement).  Initial values come from the environment, read ONCE per process: FITGNN_GEMM_WS,
 * FITGNN_HEAD_BULK, FITGNN_AGG_WIDE, FITGNN_GEMM_WIDE, FITGNN_GEMM_PAIR, FITGNN_GEMM_PAIR_WS (0 = CTA pairs never keep their
 * weights resident), FITGNN_GEMM_PREFETCH (1 = the TMA producer prefetches the next m-block's A rows into L2; measured
 * slower), FITGNN_SM_RESERVE (SMs the persistent GEMM grids leave free for a concurrent exchange kernel).
 * name = the lower-case suffix ("gemm_pair", ...).  gemm_debug (no environment variable, default 0): bit 0 = GEMM epilogues
 * skip their TMA stores (scripts/bench_*epilogue_cost.py only). */
int fitgnn_tuning_set(const char* name, int value);
int fitgnn_tuning_get(const char* name, int* value);

/* ------------------------------------------------------------------------------------------
 * Generic per-call CSR (drop-in GCNConv path).  Replaces gcn_norm inside GCNConv.__call__
 * (call sites network.py:31,60,90,126,161,197): existing self loops are dropped, one loop per
 * node is added, deg = in-degree incl. the loop, duplicate edges count twice.
 * edge_index is the reference's [2,E] int64 COO (row 0 = source, row 1 = target).
 * nnz = (E - #self loops) + n is returned by the plan call in *host_nnz.
 * ---------------------------------------------------------------------------------------- */
size_t fitgnn_csr_workspace_bytes(int64_t E, int64_t n);
int fitgnn_csr_plan(const int64_t* edge_index, int64_t E, int64_t n, void* ws, size_t ws_bytes,
                    int64_t* host_nnz, void* stream);
int fitgnn_csr_fill(int64_t n, void* ws, size_t ws_bytes, int32_t* rowptr /*[n+1]*/,
                    int32_t* col /*[nnz]*/, float* dinv /*[n]*/, void* stream);
/* Raw per-call CSR (drop-in SAGEConv path): the edges exactly as given — self loops kept, none added, duplicates kept
 * (each occurrence is one entry).  Same workspace as fitgnn_csr_plan (fitgnn_csr_workspace_bytes); *host_nnz = E.  Rows are
 * targets, entries in ascending column order inside a row.  No dinv. */
int fitgnn_csr_raw_plan(const int64_t* edge_index, int64_t E, int64_t n, void* ws, size_t ws_bytes,
                        int64_t* host_nnz, void* stream);
int fitgnn_csr_raw_fill(int64_t n, void* ws, size_t ws_bytes, int32_t* rowptr /*[n+1]*/, int32_t* col /*[nnz]*/,
                        void* stream);

/* ------------------------------------------------------------------------------------------
 * Pack builder.  Replaces coarsening_classification / coarsening_regression's per-cluster
 * loop (utils.py:186-267, :269-350, :417-501, :503-584) plus neighbour()/nodes_2_neighbours()
 * (utils.py:52-62) and Data.subgraph (utils.py:248).
 * part[v] = index of v's subgraph in the reference's subgraph_list order.
 * FITGNN_MODE_CLUSTER additionally needs the coarsened adjacency pattern Ac as CSR over the
 * same cluster ids (from fitgnn_project_adj_*), i.e. `adj = Gc.A` at utils.py:160,228.
 * ---------------------------------------------------------------------------------------- */
size_t fitgnn_pack_workspace_bytes(int64_t E, int64_t N, int64_t k, int mode, int64_t ac_nnz);
int fitgnn_pack_plan(const int64_t* edge_index, int64_t E, int64_t N, const int32_t* part, int64_t k,
                     int mode, const int32_t* ac_rowptr, const int32_t* ac_col, int64_t ac_nnz,
                     void* ws, size_t ws_bytes, fitgnn_plan* host_plan, void* stream);
/* `out` holds caller-allocated device arrays sized from host_plan (the const is cast away); ws is the
 * workspace the plan call used, ws2 a second one of host_plan->fill_ws_bytes (may be null when 0).
 * edge_index / part / ac_* passed to the plan call must still be alive. */
int fitgnn_pack_fill(const fitgnn_plan* host_plan, const fitgnn_pack* out, void* ws, size_t ws_bytes,
                     void* ws2, size_t ws2_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Segmented symmetric-normalised SpMM.  Replaces MessagePassing.propagate + bias (+ F.elu)
 * inside GCNConv (network.py:31-32):
 *   Y[i,:] = act( sum_{e in row r_i} dinv[r_i]*dinv[col_e] * X[src(col_e), :] + bias )
 * r_i = out_rows[i] (or i when out_rows is null, n_out = n_rows); src(c) = src_index[c] (gid
 * de-duplication) or c when src_index is null.  width % 4 == 0, ldx % 4 == 0, ldy % 4 == 0,
 * 16-byte aligned bases.  If y_lo is non-null Y is written as a bf16 hi/lo split instead of fp32:
 * y = bf16 hi plane, y_lo = bf16 lo plane (both [n_out, ldy] bf16) feeding FITGNN_GEMM_BF16X3.
 * ---------------------------------------------------------------------------------------- */
int fitgnn_spmm_symnorm(const int32_t* rowptr, const int32_t* col, const float* dinv,
                        const float* X, int64_t ldx, int width, const int32_t* src_index,
                        const float* bias, int act, const int32_t* out_rows, int64_t n_out,
                        void* Y, void* Y_lo, int64_t ldy, void* stream);
/* Mean aggregation of SAGEConv (PyG SAGEConv, aggr='mean', root_weight=True):  out_i = lin_l(mean_j x_j) + lin_r(x_i).
 * r_i = out_rows[i] (or i), src(c) = src_index[c] (or c).  skip_self != 0: the entry col == r_i (the one self entry of a
 * pack row) is neither summed nor counted; otherwise every entry is a neighbour.  A row without neighbours has mean 0.
 * The sum runs in CSR order (one fmaf chain per element) and is divided by the neighbour count (correctly rounded), so the
 * result is independent of out_rows / src_index.  src_scale (device, indexed by column, may be NULL): the sum is weighted by
 * src_scale[col_e] and NOT divided — with the reversed CSR and src_scale = 1/count this is the transposed mean operator.
 * Y as fitgnn_spmm_symnorm: fp32, or bf16 hi/lo planes when Y_lo != NULL.
 * concat (aggregate-first):  Y[i] = [ mean X[src(col_e), 0:width] | X[src(r_i), 0:width] ], the second half starting at
 *   column `half` (>= width); columns [width, half) and [half + width, 2*half) are written as zeros.  This is the A operand
 *   of ONE transform against [W_l | W_r] (K = 2*half), with lin_l.bias and the activation in its epilogue.
 * root (transform-first, after Z = X·[W_l ; W_r]^T):
 *   Y[i] = act( mean Z[src(col_e), 0:width] + Z[src(r_i), root_off : root_off + width] + bias ). */
int fitgnn_spmm_mean_concat(const int32_t* rowptr, const int32_t* col, const float* X, int64_t ldx, int width, int half,
                            const int32_t* src_index, const float* src_scale, int skip_self, const int32_t* out_rows,
                            int64_t n_out, void* Y, void* Y_lo, int64_t ldy, void* stream);
int fitgnn_spmm_mean_root(const int32_t* rowptr, const int32_t* col, const float* Z, int64_t ldz, int width,
                          int64_t root_off, const int32_t* src_index, const float* src_scale, int skip_self,
                          const float* bias, int act, const int32_t* out_rows, int64_t n_out, void* Y, void* Y_lo,
                          int64_t ldy, void* stream);
/* The same aggregation (no bias / activation, every row an output row) for a GROUP-ALIGNED pack
 * (fitgnn_pack_align_*): every CSR entry of a row lies in the row's own group of `group` = 32 rows, so one warp stages
 * the group's source rows in shared memory once and HBM sees every byte once.  width <= 128.  Results are bit-identical
 * to fitgnn_spmm_symnorm.  FITGNN_EUNSUP for other shapes (callers fall back to fitgnn_spmm_symnorm); entries that
 * point outside their group are a precondition violation (they are wrapped into the group, never out of bounds). */
int fitgnn_spmm_symnorm_grouped(const int32_t* rowptr, const int32_t* col, const float* dinv,
                                const float* X, int64_t ldx, int width, const int32_t* src_index,
                                int64_t n_rows, int group, void* Y, void* Y_lo, int64_t ldy,
                                int fill_pad, float pad_value, void* stream);
/* fill_pad != 0 (bf16 planes with ldy == width + 4 only, ignored otherwise): the four pad columns of every row are written
 * as well — hi[:, width] = pad_value, all other pad elements 0 — so that the planes are written in whole 32-byte sectors. */
/* The same aggregation written as ONE fp16 plane [n_rows, ldy] (ldy in elements; fp32 sums, one saturating rounding): the A
 * operand of the first transform when the whole forward runs on fp16 planes (PackedForward(precision="fp16")).  fill_pad as
 * above: Y[:, width] = pad_value, the other three pad elements 0, when ldy == width + 4. */
int fitgnn_spmm_symnorm_grouped_f16(const int32_t* rowptr, const int32_t* col, const float* dinv,
                                    const float* X, int64_t ldx, int width, const int32_t* src_index,
                                    int64_t n_rows, int group, void* Y, int64_t ldy, int fill_pad,
                                    float pad_value, void* stream);
/* The same aggregation (every row an output row) with SHARED-MEMORY STAGING of the sources: blk_ptr[n_blk + 1] (device)
 * cuts the pack rows into consecutive blocks that are closed under adjacency (unions of whole subgraphs, e.g. from
 * sub_ptr); a CTA stages a block's source rows (through src_index when given) in shared memory once and all rows of the
 * block aggregate from there, so HBM / L2 see every source row once instead of once per CSR entry — the kernel for packs
 * whose rows have many entries (cluster_node subgraphs, utils.py:190-233: ~25 per row at ogbn-products scale).  Any
 * width (wide rows go in 64-column slices); blocks beyond the staging capacity are read from global memory.
 * Bit-identical to fitgnn_spmm_symnorm.  Entries leaving their block are a precondition violation. */
int fitgnn_spmm_symnorm_blocked(const int32_t* rowptr, const int32_t* col, const float* dinv,
                                const float* X, int64_t ldx, int width, const int32_t* src_index,
                                const int32_t* blk_ptr, int64_t n_blk, const int32_t* row_order,
                                const float* bias, int act, void* Y, void* Y_lo, int64_t ldy, void* stream);
/* row_order (device, [n_rows], may be NULL = identity): a permutation of the pack rows that keeps every block's rows
 * together (positions blk_ptr[b]..blk_ptr[b+1] hold block b's rows) — e.g. sorted by row length inside each block, so
 * that the rows a warp works on at the same time have similar lengths.  Results do not depend on it. */
/* The same aggregation for DENSE blocks on the tensor cores: inside a block Â = D·M·D with M the 0/1 (small-integer)
 * adjacency — exact in bf16 — so every 128 x 128 piece of M times the block's D·X rows (bf16 hi/lo planes, 2^-17) is a small
 * dense MMA with fp32 accumulation; per CSR entry nothing is gathered at all.  For cluster_node packs (utils.py:190-233,
 * ~25 % dense subgraphs).  Sums run in MMA order: results agree with fitgnn_spmm_symnorm to ~1e-6 relative, not bit for bit. */
int fitgnn_spmm_symnorm_mma(const int32_t* rowptr, const int32_t* col, const float* dinv,
                            const float* X, int64_t ldx, int width, const int32_t* src_index,
                            const int32_t* blk_ptr, int64_t n_blk, const float* bias, int act,
                            void* Y, void* Y_lo, int64_t ldy, void* stream);
/* Same with the high-degree rows split across a CTA: hub_list (from fitgnn_spmm_hubs) holds the output
 * indices i whose row has >= hub_deg entries; the warp-per-row pass skips them. */
int fitgnn_spmm_hubs(const int32_t* rowptr, const int32_t* out_rows, int64_t n_out, int hub_deg,
                     int32_t* hub_list /*[hub_cap]*/, int32_t* hub_count /*[1] device*/, int hub_cap,
                     void* stream);
int fitgnn_spmm_symnorm_hub(const int32_t* rowptr, const int32_t* col, const float* dinv,
                            const float* X, int64_t ldx, int width, const int32_t* src_index,
                            const float* bias, int act, const int32_t* out_rows, int64_t n_out,
                            void* Y, void* Y_lo, int64_t ldy, const int32_t* hub_list, int n_hub,
                            int hub_deg, void* stream);

/* Same with a hub list whose LENGTH lives on the device (hub_count as written by fitgnn_spmm_hubs; at most hub_cap entries
 * are used, so hub_cap must bound the number of hub rows: nnz / hub_deg + 1 always does): no host synchronisation between
 * finding the hubs and using them (fitgnn_gcn_forward, CUDA-graph capture). */
int fitgnn_spmm_symnorm_devhub(const int32_t* rowptr, const int32_t* col, const float* dinv,
                               const float* X, int64_t ldx, int width, const int32_t* src_index,
                               const float* bias, int act, const int32_t* out_rows, int64_t n_out,
                               void* Y, void* Y_lo, int64_t ldy, const int32_t* hub_list,
                               const int32_t* hub_count /*[1] device*/, int hub_cap, int hub_deg, void* stream);

/* ------------------------------------------------------------------------------------------
 * Dense transform.  Replaces GCNConv.lin / lt1 (F.linear, network.py:31,34):
 *   Y[M,N] = act( A[M,K] · W[N,K]^T + bias[N] ),  W laid out as lin.weight ([out,in] row-major).
 * FITGNN_GEMM_FP32: A, W fp32.   FITGNN_GEMM_BF16X3: A_hi/A_lo and W_hi/W_lo are bf16 planes
 * (see fitgnn_split_bf16); K-extent padded to a multiple of 8 with zeros by the caller.
 * head != IDENTITY applies a row-wise (log-)softmax over the N outputs (N <= 256 for BF16X3, any N for FP32), after act.
 * Only rows [0, M) of Y are written, and of them columns [0, N) plus, with BF16X3 when Y (and Y_lo) are 16-byte aligned
 * with a pitch of a multiple of 16 bytes (the TMA-store path), zeros up to the next 16-byte boundary: [N, pad4(N)) of an
 * fp32 output, [N, pad8(N)) of both split planes (which makes them the zero K-padding of the next product's operand).
 * Every other pitch column keeps its contents.  The operands are read only in their first K columns and (W) first N
 * rows; the pitch beyond them may hold anything.
 * ---------------------------------------------------------------------------------------- */
int fitgnn_gemm_bias_act(int precision, const void* A, const void* A_lo, int64_t lda,
                         const void* W, const void* W_lo, int64_t ldw, const float* bias,
                         int64_t M, int K, int N, int act, int head, float* Y, int64_t ldy,
                         void* stream);
/* Same, with the result written as bf16 hi/lo planes (Y = hi, Y_lo = lo, both [M, ldy] bf16) ready to be the A
 * operand of the next FITGNN_GEMM_BF16X3 call; Y_lo == NULL means fp32 output as above.  BF16X3 only, no head. */
int fitgnn_gemm_bias_act_split(int precision, const void* A, const void* A_lo, int64_t lda,
                               const void* W, const void* W_lo, int64_t ldw, const float* bias,
                               int64_t M, int K, int N, int act, int head, void* Y, void* Y_lo,
                               int64_t ldy, void* stream);
/* One fused GCN layer, aggregate-first (replaces GCNConv.__call__ + F.elu, network.py:31-32, for feature widths <= 128):
 *   Y[i,:] = act( (Â · X[src_index])[r_i,:] · W^T + bias ),  r_i = out_rows[i] or i
 * The A operand of the tensor-core transform is produced in-kernel by gather warps walking the pack CSR, so there is
 * no separate SpMM launch and no HBM round trip for Â·X.  W_hi/W_lo: bf16 planes [N, ldw] with K padded to 8.
 * Y fp32 [n_out, ldy], or bf16 hi/lo planes when Y_lo != NULL.  Returns FITGNN_EUNSUP for ineligible shapes
 * (width > 128, N <= 128, too few row blocks): callers then use fitgnn_spmm_symnorm + fitgnn_gemm_bias_act. */
int fitgnn_gcn_layer_fused(const int32_t* rowptr, const int32_t* col, const float* dinv, const float* X,
                           int64_t ldx, int width, const int32_t* src_index, const int32_t* out_rows,
                           int64_t n_out, const void* W_hi, const void* W_lo, int64_t ldw,
                           const float* bias, int N, int act, void* Y, void* Y_lo, int64_t ldy,
                           void* stream);
/* ------------------------------------------------------------------------------------------
 * Group-aligned packs and the aggregation fused into the transform's epilogue.
 * Between two conv layers the reference runs  x = F.elu(conv_i(x)); ...; conv_{i+1}(x)  (network.py:31-33), i.e. the
 * activated output of one transform is immediately propagated over the same block-diagonal adjacency.  When every
 * subgraph has at most 32 rows the pack can be re-laid-out so that no subgraph straddles a multiple of 32 rows
 * (fitgnn_pack_align_*); a row's neighbours are then rows of its own group of 32, which is exactly one TMEM lane
 * quadrant / one epilogue warp of the tensor-core transform, and the propagate step becomes register shuffles inside
 * that epilogue (fitgnn_gcn_transform_aggregate) instead of an SpMM launch with an HBM round trip.
 *
 * Placement policy: FITGNN_ALIGN_IN_ORDER keeps the subgraph order (greedy; a group is closed with padding when the next
 *   subgraph does not fit); FITGNN_ALIGN_BY_DEGREE places subgraphs by (largest non-self row degree desc, size desc, index
 *   asc) and fills the gap at a group's tail from the other end of that order — the fused aggregation loops to the largest
 *   row degree among a warp's 32 rows, so similar degrees belong together, and low-degree fillers replace the padding.
 * fitgnn_pack_align_plan: new_sub_ptr[s] = first aligned row of subgraph s (device, [n_sub+1], last = aligned row
 *   count, also returned in *host_n_rows_aligned); *host_alignable = 0 when some subgraph has more than `group` rows.
 *   Workspace: fitgnn_pack_align_workspace_bytes(n_sub, 0) for the plan, (n_sub, n_rows_aligned) for the fill.
 * fitgnn_pack_align_fill: fills the caller-allocated aligned pack `out` (n_rows = aligned row count; nnz, n_sub,
 *   n_core, n_src as `in`): padding rows are empty CSR rows with dinv = 0, they belong to the subgraph they follow.
 *   orig_row[aligned row] = row of `in` (-1 for padding), new_of_old[row of in] = aligned row,
 *   agg_desc[aligned row] = bits [0,4): number c <= 12 of non-self CSR entries, bits [4+5j, 9+5j): row-in-group of the
 *   j-th one (duplicates kept).  *host_flags: bit 0 = a row has more than 12 non-self entries (descriptor truncated:
 *   do not use the fused aggregation), bit 1 = a row without self loop, bit 2 = an entry leaves its subgraph.
 *   In the aligned pack sub_ptr[s] is the first row of subgraph s (not monotone under BY_DEGREE), sub_ptr[n_sub] the
 *   aligned row count.  group must be 32.
 * ---------------------------------------------------------------------------------------- */
enum { FITGNN_ALIGN_IN_ORDER = 0, FITGNN_ALIGN_BY_DEGREE = 1 };
size_t fitgnn_pack_align_workspace_bytes(int64_t n_sub, int64_t n_rows_aligned);
int fitgnn_pack_align_plan(const fitgnn_pack* in, int group, int policy, int32_t* new_sub_ptr,
                           int64_t* host_n_rows_aligned, int* host_alignable, void* ws, size_t ws_bytes,
                           void* stream);
int fitgnn_pack_align_fill(const fitgnn_pack* in, const int32_t* new_sub_ptr, int group,
                           int64_t n_rows_aligned, const fitgnn_pack* out, int32_t* orig_row,
                           int32_t* new_of_old, uint64_t* agg_desc, int* host_flags, void* ws,
                           size_t ws_bytes, void* stream);
/* G = Â_local · act(A·W^T + bias) on a group-aligned pack (FITGNN_GEMM_BF16X3 operands, N > 128):
 *   G[r,:] = dinv[r] * ( dinv[r]*h[r,:] + sum_{c in agg_desc(r)} dinv[c]*h[c,:] ),  h = act(A·W^T + bias)
 * = the next GCNConv's propagate (gcn_norm weights, self loop included) applied to this layer's activated output.
 * Y fp32 [M, ldy], or bf16 hi/lo planes when Y_lo != NULL.  Padding rows (dinv = 0) are written as zeros; the
 * padding rows of A must hold finite values.  defer_row_scale != 0 stores the sum WITHOUT the leading dinv[r]: a row
 * scaling commutes with the next transform, whose epilogue applies it for free (fitgnn_gemm_rowscale_bias_act_split). */
int fitgnn_gcn_transform_aggregate(const void* A_hi, const void* A_lo, int64_t lda, const void* W_hi,
                                   const void* W_lo, int64_t ldw, const float* bias, int64_t M, int K,
                                   int N, int act, const uint64_t* agg_desc, const float* dinv,
                                   int defer_row_scale, void* Y, void* Y_lo, int64_t ldy, void* stream);
/* fitgnn_gemm_bias_act_split with a per-row factor:  Y = head(act(row_scale[m] * (A·W^T)[m,:] + bias)).
 * row_scale may be NULL (= 1); non-NULL needs FITGNN_GEMM_BF16X3.  A head normalises the scaled logits. */
int fitgnn_gemm_rowscale_bias_act_split(int precision, const void* A, const void* A_lo, int64_t lda,
                                        const void* W, const void* W_lo, int64_t ldw,
                                        const float* row_scale, const float* bias, int64_t M, int K,
                                        int N, int act, int head, void* Y, void* Y_lo, int64_t ldy,
                                        void* stream);
/* FITGNN_GEMM_FP16X2 — a cheaper operand format for the HIDDEN STATE, opt-in (PackedForward(precision="fp16x2")):
 * the A operand is ONE fp16 plane (11-bit significand, 2 bytes per element instead of the 4 of a bf16 hi/lo pair), W an fp16
 * hi/lo pair (fitgnn_split_f16: 22 bits), two MMAs per k-step (A*W_hi + A*W_lo) instead of three, fp32 accumulation.
 * Relative error of a product: 2^-11 per A element (measured end to end on the products workload: 1.6e-5 of the 1e-3 bound,
 * profiles/r2_precision_study.md); whether that is acceptable depends on the checkpoint, hence not the default.
 *   fitgnn_gemm_f16: Y = head(act(row_scale * (A·W^T) + bias)); out_f16 != 0 stores Y as ONE fp16 plane [M, ldy] (the next
 *     FP16X2 product's A; no head / row map then), else fp32 [M, ldy] (row_map as in fitgnn_gemm_head_rows, may be NULL).
 *   fitgnn_gcn_transform_aggregate_f16: fitgnn_gcn_transform_aggregate with an fp16-plane OUTPUT; the input is a bf16
 *     hi/lo pair (in_f16 = 0, W = bf16 planes: the first layer) or an fp16 plane (in_f16 = 1, A_lo = NULL, W = fp16 planes).
 *     agg_desc may be NULL: the plain transform act(A·W^T + bias) into an fp16 plane (classic schedule, first layer).
 *   fitgnn_spmm_symnorm_f16: fitgnn_spmm_symnorm_hub / _devhub on ONE fp16 plane in and out (ldx / ldy in elements, fp32
 *     sums): the later layers' aggregation of the classic schedule, half the gathered bytes.  hub_count (device) may be
 *     NULL: hub_cap is then the host-known number of hub rows (0 = none).
 *   fitgnn_split_f16: fp32 -> fp16 hi/lo planes (lo may be NULL: the hi plane only); values beyond +-65504 saturate.
 * W_lo = NULL in fitgnn_gemm_f16 / fitgnn_gcn_transform_aggregate_f16 (in_f16 = 1) selects ONE fp16 weight plane as well
 * (PackedForward(precision="fp16") for the hidden -> hidden transforms): one MMA per k-step, 2^-11 per element on both
 * operands (measured end to end: 1.8e-5 of the largest logit against 1.6e-5 with hi/lo weights, profiles/r2_precision_study.md),
 * and for K <= 512 the CTA-pair kernel keeps each CTA's half of the 256-row weight block resident in shared memory
 * (W-stationary pairs: only A streams; tuning switch gemm_pair_ws = 0 restores the streaming plan).
 * Every fp16-plane output of these kernels is rounded to nearest once and saturates: a value beyond +-65504 is stored as
 * +-65504, never as inf. */
int fitgnn_split_f16(const float* X, int64_t ldx, int64_t rows, int cols, void* hi, void* lo, int64_t ldo, void* stream);
int fitgnn_gemm_f16(const void* A, int64_t lda, const void* W_hi, const void* W_lo, int64_t ldw,
                    const float* row_scale, const float* bias, int64_t M, int K, int N, int act, int head,
                    void* Y, int64_t ldy, int out_f16, const int32_t* row_map, void* stream);
int fitgnn_spmm_symnorm_f16(const int32_t* rowptr, const int32_t* col, const float* dinv, const void* X, int64_t ldx,
                            int width, const int32_t* src_index, const float* bias, int act, const int32_t* out_rows,
                            int64_t n_out, void* Y, int64_t ldy, const int32_t* hub_list, const int32_t* hub_count,
                            int hub_cap, int hub_deg, void* stream);
/* A whole GCNConv of a group-aligned pack in ONE kernel (network.py:31-32, `x = F.elu(conv(x, edge_index))`, for the layers
 * after the first; the fp16 hidden state): Y = act(Â·(A·W^T) + bias) with Â the pack's normalised adjacency.  The aggregation
 * runs in the transform's epilogue on the raw fp32 accumulators (thread = row, a warp = one aligned group, neighbours are
 * other lanes), then bias and activation; A and Y are fp16 planes [M, lda] / [M, ldy], W fp16 planes (W_lo may be NULL: one
 * plane).  For K > 128 and M >= 4096 this is the CTA-pair kernel (W-stationary when the weights fit), whose tensor-bound
 * main loop hides the exchange-heavy epilogue; PackedForward(precision="fp16" / "fp16x2") uses it for every layer after the
 * first (schedule: spmm0 -> transform -> [conv]* -> head).  A padding row (dinv = 0) is NOT written as zeros: it holds
 * act(bias) rounded to fp16 (0 without a bias), because the trailing dinv[r] scales the aggregate and not the bias. */
int fitgnn_gcn_conv_aligned_f16(const void* A, int64_t lda, const void* W_hi, const void* W_lo, int64_t ldw,
                                const float* bias, int64_t M, int K, int N, int act, const uint64_t* agg_desc,
                                const float* dinv, void* Y, int64_t ldy, void* stream);
/* fitgnn_gemm_head_rows_peers with an fp16-plane A operand (FITGNN_GEMM_FP16X2) */
int fitgnn_gemm_f16_head_rows_peers(const void* A, int64_t lda, const void* W_hi, const void* W_lo, int64_t ldw,
                                    const float* bias, int64_t M, int K, int N, int act, int head,
                                    const int32_t* row_map, float* const* host_peer_bases, int n_peers,
                                    int64_t ldy, void* stream);
/* SAGEConv on the fp16 hidden state (PackedForward(precision="fp16x2" / "fp16") for a SAGE state_dict):
 *   fitgnn_spmm_mean_f16: the mean aggregation of fitgnn_spmm_mean_concat with X and Y ONE fp16 plane each (ldx / ldy in
 *     elements; width, half, ldx, ldy multiples of 8, 16-byte aligned planes).  One 16-byte load of 8 halfs per lane and source
 *     row, fp32 sums in CSR order, one division, one saturating rounding.  concat != 0: Y[i] = [mean | root] as the concat form
 *     (ldy >= 2*half); concat = 0: the mean alone, Y[i] = mean, columns [width, half) zero (ldy >= half).  skip_self, src_index
 *     and out_rows as fitgnn_spmm_mean_concat (no src_scale); results are bit-identical across out_rows / src_index.
 *   fitgnn_spmm_mean_root_f16: fitgnn_spmm_mean_root (fp32 Z, no src_scale) whose output is ONE fp16 plane [n_out, ldy].
 *   fitgnn_gemm_f16_2seg: fitgnn_gemm_f16 (no row scale, head or row map) whose A operand is two fp16 planes side by side in K:
 *     columns [0, K0) are A0 (a0_cols <= K0 columns of pitch lda0, zero beyond), columns [K0, K) are A1 (K - K0 columns of
 *     pitch lda1).  K0 is a multiple of 64 (the k-block).  Neither plane is read beyond its width.  Both planes have M rows.
 *     With A0 = the mean plane and A1 = the hidden state itself this is lin_l(mean h) + lin_r(h) against
 *     W = [W_l | 0 | W_r] (K0 = hidden rounded up to 64) without a concatenated operand.  Bit-identical to fitgnn_gemm_f16 on
 *     the materialised [A0 | 0 | A1]: same plans, same MMAs in the same order. */
int fitgnn_spmm_mean_f16(const int32_t* rowptr, const int32_t* col, const void* X, int64_t ldx, int width, int half,
                         const int32_t* src_index, int skip_self, int concat, const int32_t* out_rows, int64_t n_out, void* Y,
                         int64_t ldy, void* stream);
int fitgnn_spmm_mean_root_f16(const int32_t* rowptr, const int32_t* col, const float* Z, int64_t ldz, int width,
                              int64_t root_off, const int32_t* src_index, int skip_self, const float* bias, int act,
                              const int32_t* out_rows, int64_t n_out, void* Y, int64_t ldy, void* stream);
int fitgnn_gemm_f16_2seg(const void* A0, int64_t lda0, int a0_cols, int K0, const void* A1, int64_t lda1, const void* W_hi,
                         const void* W_lo, int64_t ldw, const float* bias, int64_t M, int K, int N, int act, void* Y,
                         int64_t ldy, int out_f16, void* stream);
int fitgnn_gcn_transform_aggregate_f16(int in_f16, const void* A_hi, const void* A_lo, int64_t lda, const void* W_hi,
                                       const void* W_lo, int64_t ldw, const float* bias, int64_t M, int K, int N,
                                       int act, const uint64_t* agg_desc, const float* dinv, int defer_row_scale,
                                       void* Y, int64_t ldy, void* stream);
/* fitgnn_gemm_bias_act (BF16X3) whose output row m is written to Y row row_map[m] and skipped when row_map[m] < 0:
 * drops the padding rows of an aligned pack / scatters lt1's output (network.py:34-35) straight into the caller's
 * row order.  When ldy is N rounded up to a multiple of 4, the pitch-padding columns [N, ldy) of written rows are
 * zero-filled, whichever store path runs (narrow heads write whole rows with bulk copies, the others per row); otherwise
 * they are left untouched. */
int fitgnn_gemm_head_rows(const void* A_hi, const void* A_lo, int64_t lda, const void* W_hi,
                          const void* W_lo, int64_t ldw, const float* bias, int64_t M, int K, int N,
                          int act, int head, const int32_t* row_map, float* Y, int64_t ldy, void* stream);
/* ------------------------------------------------------------------------------------------
 * Multi-GPU output exchange fused into the head (one process per GPU on one NVLink/NVSwitch box).
 * The reference is single-device (SURVEY §2a); with the subgraphs sharded over N ranks the only
 * inference-path exchange is the gather of the core-node outputs (SURVEY §8e).
 * fitgnn_gemm_head_rows_peers = fitgnn_gemm_head_rows whose output row m is stored to
 *   host_peer_bases[p] + row_map[m] * ldy   for every p in [0, n_peers)
 * i.e. into the same slot of every rank's gather buffer (peer-mapped device pointers, the stores travel
 * over NVLink while the kernel computes), so no all-gather follows the head: a barrier among the ranks
 * (stream-ordered, e.g. a one-element all-reduce) is all that remains.  host_peer_bases is a HOST array.
 * fitgnn_peer_alloc/open/close/free provide such buffers: cudaMalloc'ed (zero-filled) memory exported as a
 * 64-byte CUDA IPC handle and imported by the other ranks (peer access is enabled on import).
 * ---------------------------------------------------------------------------------------- */
int fitgnn_gemm_head_rows_peers(const void* A_hi, const void* A_lo, int64_t lda, const void* W_hi,
                                const void* W_lo, int64_t ldw, const float* bias, int64_t M, int K,
                                int N, int act, int head, const int32_t* row_map,
                                float* const* host_peer_bases, int n_peers, int64_t ldy, void* stream);
/* fitgnn_peer_push: copy `bytes` (multiple of 16) from this rank's slot `src` to host_dst[0..n_dst) (the same slot in
 * the peers' buffers) with a small kernel of n_ctas CTAs (0 = 16) that streams the slot through shared memory with bulk
 * copies — meant for a side stream, behind the next step's compute (dist.PeerGather 'push' exchange). */
int fitgnn_peer_push(const void* src, void* const* host_dst, int n_dst, size_t bytes, int n_ctas, void* stream);
int fitgnn_peer_alloc(size_t bytes, void** dev_ptr, uint8_t* handle_out /*[64] host*/);
int fitgnn_peer_open(const uint8_t* handle /*[64] host*/, void** dev_ptr);
int fitgnn_peer_close(void* dev_ptr);
int fitgnn_peer_free(void* dev_ptr);
/* fp32 [rows, cols] (ld = ldx) -> bf16 hi/lo planes [rows, ldo] (columns >= cols zero filled) */
int fitgnn_split_bf16(const float* X, int64_t ldx, int64_t rows, int cols, void* hi, void* lo,
                      int64_t ldo, void* stream);

/* ------------------------------------------------------------------------------------------
 * The whole forward in one call.  Replaces, for every subgraph of the pack at once, Classify_node.forward /
 * Regress_node.forward (network.py:29-35, :58-64; Net1 / Net2 inference.py:87-93, :110-116) as driven by
 * node_infer_Gs_GD (run.py:59-77) and the per-query loop (inference.py:672-688):
 *   n_layers x ( GCNConv -> ELU ) -> lt1 -> head, evaluated on the pack, returning the CORE rows (the rows the callers
 *   read, run.py:73) in pack order: out[i, :] belongs to pack row core_rows[i] = node gid[core_rows[i]].
 * weights: the model's parameters as the reference's state_dict holds them (conv.{i}.lin.weight [out, in] row-major,
 *   conv.{i}.bias [out], lt1.weight [n_classes, hidden], lt1.bias) — DEVICE pointers; conv_weight / conv_bias are HOST
 *   arrays of n_layers device pointers.
 * X: de-duplicated feature table [n_src, ldx] fp32 (every node once, + one C·X row per cluster in cluster mode), ldx a
 *   multiple of 4 and >= in_features rounded up to 4, padding columns zero.
 * precision: FITGNN_GEMM_BF16X3 (tensor cores, hidden %% 8 == 0) or FITGNN_GEMM_FP32.  head: FITGNN_HEAD_*.
 * Schedule: layer 0 transform-first on the de-duplicated rows when in_features > hidden, else aggregate-first; later
 *   layers aggregate-first; the last layer and the head only on the core rows.  Stream-ordered, no host synchronisation,
 *   no allocation (workspace of fitgnn_gcn_forward_workspace_bytes bytes, 256-byte aligned), CUDA-graph capturable.
 * ---------------------------------------------------------------------------------------- */
typedef struct fitgnn_weights {
  int n_layers;                     /* args.num_layers1 (network.py:11) */
  int in_features, hidden, n_classes;
  const float* const* conv_weight;  /* host array [n_layers] of device pointers */
  const float* const* conv_bias;    /* host array [n_layers] of device pointers (an entry may be NULL) */
  const float* lt1_weight;          /* device [n_classes, hidden] */
  const float* lt1_bias;            /* device [n_classes] or NULL */
} fitgnn_weights;
size_t fitgnn_gcn_forward_workspace_bytes(const fitgnn_pack* pack, const fitgnn_weights* weights, int precision);
int fitgnn_gcn_forward(const fitgnn_pack* pack, const float* X, int64_t ldx, const fitgnn_weights* weights,
                       int head, int precision, float* out /*[n_core, ld_out]*/, int64_t ld_out, void* ws,
                       size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Training path (node_train_Gs_GD run.py:177-215, node_train_Gc run.py:26-37; dropout network.py:33; Adam main.py:193-194).
 * fitgnn_gemm_tn: the weight gradient of GCNConv.lin / lt1 on the tensor cores,
 *     dW[out, in] = sum_r G[r, out] * A[r, in]        (G = gradient w.r.t. the layer's pre-activation, A = its input)
 *   both operands row-major fp32 [R, *]; internally a transposing bf16 hi/lo split (the contraction runs over the rows),
 *   a batched split-K FITGNN_GEMM_BF16X3 product and a fixed-order reduction of the partial sums (deterministic).
 * fitgnn_dropout: Y = X * mask / (1 - p), mask from Philox4x32-10 keyed by (seed, offset + element / 4): the backward
 *   regenerates the same mask from the same (seed, offset), nothing is stored.  Element index = row * cols + col.
 * fitgnn_elu_dropout_backward: GZ = G * mask / (1 - p) * act'(H) with H the activation's OUTPUT before the dropout
 *   (ELU'(z) = 1 for z > 0, else elu(z) + 1); p = 0 -> no mask; act = FITGNN_ACT_NONE -> act' = 1.
 * fitgnn_adam_step: torch.optim.Adam (no amsgrad) on a flat buffer: g += weight_decay * p; m, v moments; bias correction with
 *   `step` (1-based).
 * ---------------------------------------------------------------------------------------- */
size_t fitgnn_gemm_tn_workspace_bytes(int64_t R, int out, int in);
int fitgnn_gemm_tn(const float* G, int64_t ldg, const float* A, int64_t lda, int64_t R, int out, int in,
                   float* dW, int64_t lddw, void* ws, size_t ws_bytes, void* stream);
int fitgnn_dropout(const float* X, int64_t ldx, int64_t rows, int cols, float p, uint64_t seed,
                   uint64_t offset, float* Y, int64_t ldy, void* stream);
int fitgnn_elu_dropout_backward(const float* G, int64_t ldg, const float* H, int64_t ldh, int64_t rows,
                                int cols, int act, float p, uint64_t seed, uint64_t offset, float* GZ,
                                int64_t ldo, void* stream);
int fitgnn_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                     float beta1, float beta2, float eps, float weight_decay, int64_t step, void* stream);

/* ------------------------------------------------------------------------------------------
 * Graph-level pooling.  Replaces x[mask] + torch.cat + global_max_pool / global_mean_pool
 * (network.py:129-131, :200-202).  rows[i] selects the i-th pooled row of X (the masked rows in
 * pack order); seg_ptr[g]..seg_ptr[g+1] delimits graph g's pooled rows (batch_tensor is sorted).
 * An empty segment yields 0 (PyG scatter semantics).
 * ---------------------------------------------------------------------------------------- */
int fitgnn_segment_pool(const float* X, int64_t ldx, int width, const int32_t* rows,
                        const int32_t* seg_ptr, int64_t n_seg, int pool, float* Y, int64_t ldy,
                        void* stream);

/* ------------------------------------------------------------------------------------------
 * Coarsened-graph projection.
 * fitgnn_project_features replaces C.dot(H_feature) (utils.py:161,738,827):
 *   Xc[c,:] = fp32( sum_{j: part[j]==c, ascending j} (double)cweight[j] * X[j,:] ), fp64 accumulate.
 *   members = node ids sorted by (part, id), member_ptr[k+1] (from fitgnn_group_by_part).
 * fitgnn_project_adj_* replaces zero_diag(coarsen_matrix(W, iC)) (coarsening_utils.py:138,201-205,
 * graph_utils.py:79-87) and Gc.W.tocoo() (utils.py:745-746): the pattern of P_bin·A·P_bin^T with the
 * diagonal removed, row-major sorted COO, cnt = number of directed edges between the two clusters.
 * ---------------------------------------------------------------------------------------- */
size_t fitgnn_group_workspace_bytes(int64_t N, int64_t k);
int fitgnn_group_by_part(const int32_t* part, int64_t N, int64_t k, int32_t* members /*[N]*/,
                         int32_t* member_ptr /*[k+1]*/, void* ws, size_t ws_bytes, void* stream);
int fitgnn_project_features(const int32_t* members, const int32_t* member_ptr, int64_t k,
                            const double* cweight /*[N] by node id*/, const float* X, int64_t ldx,
                            int F, float* Xc, int64_t ldxc, void* stream);
size_t fitgnn_project_adj_workspace_bytes(int64_t E);
int fitgnn_project_adj_plan(const int64_t* edge_index, int64_t E, int64_t N, const int32_t* part,
                            int64_t k, void* ws, size_t ws_bytes, int64_t* host_nnz, void* stream);
int fitgnn_project_adj_fill(void* ws, size_t ws_bytes, int64_t k, int64_t* out_row, int64_t* out_col,
                            int32_t* out_cnt, int32_t* out_rowptr /*[k+1] or null*/, void* stream);

/* ------------------------------------------------------------------------------------------
 * Device primitives used by the builders, exported for tests.
 * ---------------------------------------------------------------------------------------- */
size_t fitgnn_sort_workspace_bytes(int64_t n);
/* ascending LSD radix sort of the low `key_bits` bits; vals may be null; sorts in place */
int fitgnn_sort_u64(uint64_t* keys, uint32_t* vals, int64_t n, int key_bits, void* ws,
                    size_t ws_bytes, void* stream);
/* exclusive prefix sum, out may alias in; out[n] (one past) receives the total when with_total */
int fitgnn_scan_i32(const int32_t* in, int32_t* out, int64_t n, int with_total, void* ws,
                    size_t ws_bytes, void* stream);
size_t fitgnn_scan_workspace_bytes(int64_t n);

#ifdef __cplusplus
}
#endif
#endif /* FITGNN_H_ */
