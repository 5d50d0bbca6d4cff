/*
 * hgr.h -- C ABI of libhgr.so: the B200 (sm_100a) embedding-propagation / loss / full-rank-eval
 * path of the SELFRec-based hypergraph-diffusion recommender.
 *
 * The reference (DanbiAubrey/Hypergraph_diffusion_for_recommendation) is pure Python and has no FFI;
 * each entry point below names the reference call site (file:line, relative to HD_SELFRec/) whose
 * library call it replaces.  INTEGRATION.md shows the ctypes binding a maintainer of the reference
 * would add at each of those call sites.
 *
 * Conventions
 *   - every function returns 0 on success or a negative hgr_status; hgr_last_error() returns a
 *     thread-local message for the last failure.  Nothing falls back to the CPU.
 *   - all pointers are DEVICE pointers owned by the caller unless a parameter says "host"; the
 *     library never allocates, frees or retains them (workspace comes from the caller, sized by the
 *     *_workspace_bytes queries).  No hidden cudaMalloc, no hidden synchronisation: every call
 *     only enqueues work on `stream` unless documented otherwise.
 *   - dense operands are fp32, row-major, contiguous [rows, D] with D in {32, 64, 128} and 16-byte
 *     aligned base pointers; indices are int32 (N < 2^31), nonzero offsets int64.
 */
#ifndef HGR_H_
#define HGR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st *hgr_stream_t; /* a cudaStream_t */

typedef enum {
    HGR_OK = 0,
    HGR_ERR_INVALID = -1,   /* bad argument (shape, dtype width, alignment, null pointer) */
    HGR_ERR_CUDA = -2,      /* a CUDA runtime call or kernel launch failed */
    HGR_ERR_UNSUPPORTED = -3,
    HGR_ERR_WORKSPACE = -4  /* caller-provided workspace too small */
} hgr_status;

const char *hgr_last_error(void);
int hgr_version(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
uint64_t hgr_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * Sparse matrix in CSR with an optional split plan for long rows.
 * Replaces the torch sparse COO tensor built by TorchGraphInterface.convert_sparse_mat_to_tensor
 * (base/torch_interface.py:8-12).  Rows longer than `chunk_nnz` nonzeros are listed in
 * `heavy_rows`; heavy row h owns chunks [heavy_chunk_ptr[h], heavy_chunk_ptr[h+1]) of `chunk_nnz`
 * consecutive nonzeros each, `chunk_owner[c]` is the h of chunk c.  n_heavy_rows == 0 disables
 * splitting (every row is then accumulated strictly sequentially, the order of the CPU oracle).
 * With `chunk_start` the chunks have explicit boundaries instead (chunk c covers nonzeros
 * [chunk_start[c], chunk_start[c + 1]) or, for the last chunk of its row, up to the row's end):
 * the window-aligned plan of hgr_window_split_count / _fill, whose chunks end where a row leaves a
 * window of the gathered table, so that a work list ordered by window keeps that window in L2.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t n_rows, n_cols;
    int64_t nnz;
    const int64_t *indptr;  /* [n_rows + 1] */
    const int32_t *indices; /* [nnz] column ids, ascending inside a row */
    const float *values;    /* [nnz] */
    int32_t chunk_nnz;
    int32_t n_heavy_rows;
    int64_t n_chunks;
    const int32_t *heavy_rows;      /* [n_heavy_rows] */
    const int64_t *heavy_chunk_ptr; /* [n_heavy_rows + 1] */
    const int32_t *chunk_owner;     /* [n_chunks] */
    /* Schedule of the propagation kernel, required whenever n_rows > 0: entry w >= 0 is unsplit row w, entry
     * w < 0 is chunk ~w of the split plan; 16 consecutive entries (D = 64) share a thread block.  Every unsplit
     * row and every chunk must appear exactly once.  graph.py bins rows by length or orders them by the window
     * of the gathered table they read; the order never changes a result bit (each row is still accumulated by
     * one row group in stored order). */
    const int32_t *work_order; /* [n_work] */
    int64_t n_work;
    const int64_t *chunk_start; /* [n_chunks] first nonzero of every chunk, or NULL: chunk k of a row starts at k * chunk_nnz */
} hgr_csr_t;

/* Row-wise epilogue fused into the propagation kernel; applied to the accumulated row `acc` in
 * this order (every stage optional):
 *   pre[row]  = acc                                   (saved for the backward pass)
 *   acc       = leaky_relu(acc, slope)                HGCNConv act, model/graph/HGNN_HD3.py:545-549
 *   acc       = LayerNorm(acc) * gamma + beta         lns[k](...), HGNN_HD3.py:421,710,714
 *   acc      += residual[row]                         "+ res" / "+ Xve", same lines
 *   acc       = (acc + sum_j addend[j][row]) * scale  layer mean/sum readout, LightGCN.py:135-136
 *   y[row]    = acc                                   (+ the same row into every gather_out table)
 */
#define HGR_MAX_ADDENDS 8
#define HGR_MAX_GATHER 8
typedef struct {
    int32_t use_leaky;
    float leaky_slope;
    const float *ln_gamma; /* [D] or NULL: no LayerNorm */
    const float *ln_beta;  /* [D] */
    float ln_eps;
    const float *residual; /* [n_rows, D] or NULL */
    int32_t n_addends;
    const float *addends[HGR_MAX_ADDENDS]; /* each [n_rows, D] */
    float scale;                           /* applied only when n_addends > 0 or scale_always != 0 */
    int32_t scale_always;
    float *pre;                            /* [n_rows, D] or NULL */
    /* Fused all-gather (multi-GPU, dist.py): the finished row is ALSO stored at row
     * gather_row_offset + row of every table in gather_out -- the gathered [world * n_loc, D] buffers of
     * all ranks, peer-mapped over NVLink (symmetric memory) -- so the exchange that follows a sharded
     * propagation rides on the kernel's own epilogue instead of a separate collective.  y may then be
     * NULL.  The caller orders the peers' reads after the kernel with a cross-rank barrier. */
    int32_t n_gather;
    float *gather_out[HGR_MAX_GATHER];
    int64_t gather_row_offset;
    /* NVSwitch multicast form of the same exchange: the MULTICAST address of the gathered table (one virtual address bound to
     * every rank's copy, NVLS).  When non-NULL a row is published with ONE multimem.st per 16 bytes and the switch replicates
     * it to all ranks, instead of n_gather unicast stores (1/world of the egress).  gather_out / n_gather are then ignored. */
    float *gather_mc;
} hgr_epilogue_t;

/* Y[n_rows, D] = epilogue(A . X[n_cols, D]).  Replaces torch.sparse.mm(adj, X)
 * (model/graph/LightGCN.py:133, HCCF.py:199, SGL.py:156-160, HGNN_HD3.py:549-553).
 * `workspace` must hold hgr_spmm_workspace_bytes(A, D) bytes (0 when the plan has no heavy rows).
 * `epi` may be NULL.  Deterministic: the same inputs give the same bits on every run. */
size_t hgr_spmm_workspace_bytes(const hgr_csr_t *A, int32_t D);
/* Window-aligned split plan (graph.py: window_split_plan).  A row is walked once in stored order; a chunk ends at nonzero j
 * when the row crosses into another window of the gathered table there (indices[j] >> window_shift differs from the previous
 * nonzero's) and the chunk already holds >= min_seg nonzeros, or when it holds max_seg nonzeros; window crossings only count in
 * rows whose first and last column lie >= min_span windows apart (a narrower row gathers from a stretch L2 holds anyway).  `_count` writes the number
 * of chunks of every row (1: the row stays whole); the host lists the rows with more than one chunk as heavy_rows, prefix-sums
 * their counts into heavy_chunk_ptr, and `_fill` writes chunk_start[heavy_chunk_ptr[h] + k] for every chunk of heavy row h.
 * The plan depends only on the sparsity pattern, never on a schedule: results stay reproducible run to run. */
int hgr_window_split_count(const int64_t *indptr, const int32_t *indices, int32_t n_rows, int32_t window_shift, int32_t min_seg,
                           int32_t max_seg, int32_t min_span, int32_t *n_seg, hgr_stream_t stream);
int hgr_window_split_fill(const int64_t *indptr, const int32_t *indices, const int32_t *heavy_rows, const int64_t *heavy_chunk_ptr,
                          int32_t n_heavy_rows, int32_t window_shift, int32_t min_seg, int32_t max_seg, int32_t min_span, int64_t *chunk_start,
                          hgr_stream_t stream);
int hgr_spmm_f32(const hgr_csr_t *A, const float *X, float *Y, int32_t D, const hgr_epilogue_t *epi,
                 void *workspace, size_t workspace_bytes, hgr_stream_t stream);

/* Y = epilogue(A . (At . X)): the node -> hyperedge -> node two-stage propagation of
 * HGCNConv.forward (model/graph/HGNN_HD3.py:540-553; 17 more copies listed in SURVEY.md 2.1).
 * `At` is the CSR of A^T (pass A itself for the symmetric normalised adjacency); `tmp` is the
 * [At->n_rows, D] hyperedge intermediate.  Workspace = max of the two stages. */
int hgr_hgconv_f32(const hgr_csr_t *A, const hgr_csr_t *At, const float *X, float *tmp, float *Y, int32_t D,
                   const hgr_epilogue_t *epi, void *workspace, size_t workspace_bytes, hgr_stream_t stream);

/* LGCN_Encoder.forward (model/graph/LightGCN.py:129-140): E^{k+1} = A E^k for k < n_layers and
 * out = mean_k E^k (sum_readout != 0: plain sum, the HCCF/SHT readout, HCCF.py:188).  `layers`
 * holds the n_layers-1 intermediate tables E^1..E^{L-1} back to back ([L-1, N, D]); the last
 * propagation never materialises E^L: its epilogue adds E^0..E^{L-1} and scales. */
int hgr_lightgcn_forward_f32(const hgr_csr_t *A, const float *E0, float *layers, float *out, int32_t n_layers,
                             int32_t D, int32_t sum_readout, void *workspace, size_t workspace_bytes,
                             hgr_stream_t stream);

/* Backward of y = LayerNorm(leaky_relu(pre)) * gamma + beta (the fused epilogue above, residual
 * excluded): dpre from dy.  dgamma/dbeta are accumulated per block into `partials`
 * ([hgr_ln_bwd_partial_rows(n_rows), 2, D]) and reduced in a fixed order by the second kernel, so
 * the result is deterministic.  gamma == NULL means "no LayerNorm" (only the leaky slope applies). */
/* y = LayerNorm(x) * gamma + beta over rows of D floats (torch.nn.LayerNorm(D), e.g. the MLP input norm of EquivSetConv,
 * model/layers/MLP.py:109-110); its backward is hgr_leaky_ln_bwd_f32 with pre = x and use_leaky = 0. */
int hgr_layer_norm_f32(const float *x, const float *gamma, const float *beta, float ln_eps, int64_t n_rows, int32_t D, float *y,
                       hgr_stream_t stream);
int32_t hgr_ln_bwd_partial_rows(int64_t n_rows);
int hgr_leaky_ln_bwd_f32(const float *pre, const float *dy, const float *gamma, float ln_eps, int32_t use_leaky,
                         float leaky_slope, int64_t n_rows, int32_t D, float *dpre, float *dgamma, float *dbeta,
                         float *partials, hgr_stream_t stream);

/* Destination of a fused all-gather (multi-GPU, dist.py) for kernels other than the propagation: row r of the producer is
 * ALSO stored at row row_offset + r of every table in `out` (the gathered [world * n_loc, D] buffers of all ranks,
 * peer-mapped over NVLink), exactly like hgr_epilogue_t::gather_out.  The caller orders the peers' reads with a
 * cross-rank barrier. */
typedef struct {
    int32_t n_gather;
    float *out[HGR_MAX_GATHER];
    int64_t row_offset;
    float *mc; /* multicast address of the gathered table, or NULL (see hgr_epilogue_t::gather_mc) */
} hgr_gather_t;

/* hgr_leaky_ln_bwd_f32 whose dpre rows -- the input of the sharded backward propagation that always follows
 * (dist.py, _DistHGConv.backward) -- are published into every rank's gathered table by the kernel that computes them. */
int hgr_leaky_ln_bwd_gather_f32(const float *pre, const float *dy, const float *gamma, float ln_eps, int32_t use_leaky,
                                float leaky_slope, int64_t n_rows, int32_t D, float *dpre, float *dgamma, float *dbeta,
                                float *partials, const hgr_gather_t *gather, hgr_stream_t stream);
/* Plain publication of owned rows x[n_rows, D] (rows that come out of a dense layer or an elementwise op): one read, one
 * 128-bit store per destination.  Replaces ncclAllGather for the exchanges no propagation kernel can carry. */
int hgr_publish_rows_f32(const float *x, int64_t n_rows, int32_t D, const hgr_gather_t *gather, hgr_stream_t stream);


/* ---------------------------------------------------------------------------------------------
 * Device construction of canonical CSR matrices (columns ascending, duplicates merged).
 * Replaces Interaction.__create_sparse_bipartite_adjacency (data/ui_graph.py:70-84),
 * Interaction.__create_sparse_interaction_matrix (data/ui_graph.py:95-112) and
 * Graph.normalize_graph_mat (data/graph.py:11-25).
 *
 * hgr_coo_to_csr: entries (rows[j], cols[j]), each of weight 1; duplicates are summed, so
 * values[p] is the multiplicity of the p-th distinct entry (scipy's csr_matrix((ones, (r, c)))).
 * `indices` and `values` need room for n_entries elements; the number of distinct entries is
 * written to the DEVICE scalar *nnz_out.  row_entries[r] (optional) = entries of row r counted
 * with duplicates = the row sum the reference normalises by.
 * hgr_bipartite_to_csr: the (U+I) x (U+I) adjacency [[0, R], [R^T, 0]] of the interaction list
 * (users[j], items[j]); indices/values need room for 2 * n_edges elements.
 * Workspace: hgr_build_csr_workspace_bytes(number of entries sorted) bytes, 256-byte aligned
 * (n_entries for hgr_coo_to_csr, 2 * n_edges for hgr_bipartite_to_csr).
 * ------------------------------------------------------------------------------------------- */
size_t hgr_build_csr_workspace_bytes(int64_t n_entries);
int hgr_coo_to_csr(const int32_t *rows, const int32_t *cols, int64_t n_entries, int32_t n_rows, int32_t n_cols,
                   int64_t *indptr, int32_t *indices, float *values, int32_t *row_entries, int64_t *nnz_out,
                   void *workspace, size_t workspace_bytes, hgr_stream_t stream);
int hgr_bipartite_to_csr(const int32_t *users, const int32_t *items, int64_t n_edges, int32_t n_users, int32_t n_items,
                         int64_t *indptr, int32_t *indices, float *values, int32_t *row_entries, int64_t *nnz_out,
                         void *workspace, size_t workspace_bytes, hgr_stream_t stream);

/* out[k] = lut[degree[k]]: the host passes lut = np.power(arange(lut_len, dtype=float32), exponent)
 * with inf -> 0 (data/graph.py:15-16), because numpy's float32 pow is not correctly rounded and the
 * reference's values are whatever the host's numpy returns.  *overflow (device int, optional) counts
 * degrees outside the table. */
int hgr_degree_scale(const int32_t *degree, int64_t n, const float *lut, int32_t lut_len, float *out, int32_t *overflow,
                     hgr_stream_t stream);

/* values[p] = (row_scale[r] * values[p]) * col_scale[c], two fp32 roundings in scipy's order:
 * d_mat_inv.dot(adj_mat).dot(d_mat_inv) (data/graph.py:18-19).  Either scale may be NULL. */
int hgr_csr_scale(const int64_t *indptr, const int32_t *indices, float *values, int32_t n_rows, const float *row_scale,
                  const float *col_scale, hgr_stream_t stream);


/* Bernoulli edge dropout with the pattern kept: SpAdjDropEdge.forward (model/graph/HCCF.py:217-226; same class in HGNN_HD3.py,
 * HGNN_HD4.py, HCCF_diffusion.py).  out[p] = keep(p) ? values[p] / keep : 0 (true division), keep(p) = floor(u + keep) != 0 in
 * fp32 with u = rand[rand_pos ? rand_pos[p] : p] (the caller's uniform numbers: replay of the reference's torch.rand(nnz) stream)
 * or, with rand == NULL, a 24-bit uniform from Philox4x32-10(seed) keyed by the entry's coordinates.  mirror != 0 keys entry
 * (r, c) with (c, r): the values of the TRANSPOSED dropped matrix on the same structurally symmetric pattern (in replay mode pass
 * the transpose permutation as rand_pos instead).  Dropped entries stay as explicit zeros: row sums are bit-identical to the
 * compacted matrix, and the split plan / schedule of the propagation kernel are reused.  seed_dev (optional, DEVICE uint64): a step
 * counter mixed into the seed at run time, so a captured CUDA graph draws a new mask at every replay. */
int hgr_drop_edges_f32(const int64_t *indptr, const int32_t *indices, const float *values, int32_t n_rows, int64_t n_cols, int64_t nnz,
                       float keep, uint64_t seed, const uint64_t *seed_dev, const float *rand, const int64_t *rand_pos, int32_t mirror,
                       float *out, hgr_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Dense learned-hyperedge propagation of HCCF: HGNNLayer.forward (model/graph/HCCF.py:206-211),
 *   edge_embeds = torch.mm(adj.T, embeds);  hyper_embeds = torch.mm(adj, edge_embeds)
 * with adj = dropout(E0 W) [n, K] and embeds [n, D].  Two tall-and-skinny products (n = users or items):
 *   hgr_tall_skinny_tn_f32    T[K, D] = H[n, K]^T . E[n, D]      every SM reduces a slice of the rows, partials added in
 *                                                               block order (deterministic); K in {32, 64, 128, 256}
 *   hgr_rows_times_small_f32  Y[n, N] = [A1[n, K1] | A2[n, K2]] . B[K1 + K2, N]   B stays in shared memory;
 *                                                               K1 + K2 <= 256, N in {32, 64, 128, 256}; A2 may be NULL
 * Forward: T = H^T E, Y = H T.  Backward: dT = H^T dY, dE = H dT, dH = [dY | E] [T^T ; dT^T].
 * fp32 FMA arithmetic; agrees with torch.mm to rounding (different summation order).
 * ------------------------------------------------------------------------------------------- */
size_t hgr_tall_skinny_workspace_bytes(int64_t n, int32_t K, int32_t D);
int hgr_tall_skinny_tn_f32(const float *H, const float *E, int64_t n, int32_t K, int32_t D, float *T, void *workspace,
                           size_t workspace_bytes, hgr_stream_t stream);
int hgr_rows_times_small_f32(const float *A1, int32_t K1, const float *A2, int32_t K2, const float *B, int32_t N, int64_t n,
                             float *Y, hgr_stream_t stream);
/* The same product with the epilogue of a Linear layer: Y = [relu]([A1 | A2] . B + bias[N]) -- nn.Linear.forward (+ F.relu) of the
 * MLP / LocalAwareEncoder input layers (model/layers/MLP.py:109-117, model/graph/HGNN_HD3.py:416) with B = weight^T, in one pass
 * instead of cuBLAS sgemm + bias kernel + ReLU kernel.  bias may be NULL. */
int hgr_rows_times_small_bias_f32(const float *A1, int32_t K1, const float *A2, int32_t K2, const float *B, int32_t N, int64_t n,
                                  float *Y, const float *bias, int32_t relu, hgr_stream_t stream);
/* ... whose finished rows are ALSO published into every rank's gathered table (sharded training: the Linear that feeds a
 * propagation, model/graph/HGNN_HD3.py:600-601, carries the exchange in its epilogue).  gather may be NULL. */
int hgr_rows_times_small_gather_f32(const float *A1, int32_t K1, const float *A2, int32_t K2, const float *B, int32_t N, int64_t n,
                                    float *Y, const float *bias, int32_t relu, const hgr_gather_t *gather, hgr_stream_t stream);
/* out = a + b on [n_rows, D] tables (the "+ res" that closes an encoder layer, model/graph/HGNN_HD3.py:419), the sum published
 * the same way.  gather may be NULL. */
int hgr_add_rows_f32(const float *a, const float *b, int64_t n_rows, int32_t D, float *out, const hgr_gather_t *gather, hgr_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * BPR + L2 loss fused with the embedding gathers (util/loss_torch.py:5-9,17-21 called from
 * model/graph/LightGCN.py:52-55, HGNN_HD3.py:339-343, HCCF.py:60).
 *   out[0] = mean_b -log(10e-6 + sigmoid(<U[u_b], I[p_b]> - <U[u_b], I[n_b]>))
 *   out[1] = reg * (||U[u]||_F + ||I[p]||_F + ||I[n]||_F) / batch_size_div
 * u, p, n are int64 [batch] (the dtype of the reference's sampler, util/sampler.py:261-263).
 * `saved` (hgr_bpr_l2_workspace_bytes(batch) bytes) carries what the backward pass needs.
 * Out-of-range indices are skipped and counted in *bad_index_count (device int, caller zeroes it).
 * Backward: d_user_tab / d_item_tab must be zero-filled by the caller; row gradients are
 * accumulated with red.global.add.f32; grad_out is the DEVICE pair (d/d out[0], d/d out[1]).
 * ------------------------------------------------------------------------------------------- */
size_t hgr_bpr_l2_workspace_bytes(int64_t batch);
int hgr_bpr_l2_fwd_f32(const float *user_tab, const float *item_tab, int64_t n_users, int64_t n_items, int32_t D,
                       const int64_t *u, const int64_t *p, const int64_t *n, int64_t batch, float reg,
                       float batch_size_div, float *out, void *saved, size_t saved_bytes, int32_t *bad_index_count,
                       hgr_stream_t stream);
int hgr_bpr_l2_bwd_f32(const float *user_tab, const float *item_tab, int64_t n_users, int64_t n_items, int32_t D,
                       const int64_t *u, const int64_t *p, const int64_t *n, int64_t batch, float reg,
                       float batch_size_div, const void *saved, const float *grad_out, float *d_user_tab,
                       float *d_item_tab, hgr_stream_t stream);
/* Sharded training (dist.py): users and items index ONE gathered table of n_rows rows (forward called with
 * user_tab == item_tab == table) and this rank needs only the gradient rows [row_lo, row_hi) it owns:
 * d_rows[(row - row_lo), :] (zero-filled by the caller).  Triples that touch no owned row are skipped. */
int hgr_bpr_l2_bwd_window_f32(const float *table, int64_t n_rows, int32_t D, const int64_t *u, const int64_t *p, const int64_t *n,
                              int64_t batch, float reg, float batch_size_div, const void *saved, const float *grad_out,
                              int64_t row_lo, int64_t row_hi, float *d_rows, hgr_stream_t stream);

/* Owner-sharded forward of the same loss (dist.py, world > 1): a rank evaluates only the triples whose USER row lies in its
 * window [own_lo, own_hi) of the gathered table and writes the four batch sums it found -- sum of -log(10e-6 + sigmoid(x)),
 * sum |u|^2, sum |p|^2, sum |n|^2, in double -- to sums[4].  The caller adds `sums` over the ranks (one all_reduce of 32
 * bytes) and calls hgr_bpr_l2_finish_f32, which turns the totals into out[0] = rec loss, out[1] = reg loss and
 * norms[3] = ||U_B||, ||P_B||, ||N_B||: the same numbers on every rank, with 1/world of the gathers of the replicated form.
 * `saved` as in hgr_bpr_l2_fwd_f32 (scratch for the per-block partial sums; nothing in it is read by the backward). */
int hgr_bpr_l2_fwd_owned_f32(const float *table, int64_t n_rows, int32_t D, const int64_t *u, const int64_t *p, const int64_t *n,
                             int64_t batch, int64_t own_lo, int64_t own_hi, double *sums, void *saved, size_t saved_bytes,
                             int32_t *bad_index_count, hgr_stream_t stream);
int hgr_bpr_l2_finish_f32(const double *sums, int64_t batch, float reg, float batch_size_div, float *out, float *norms,
                          hgr_stream_t stream);
/* Backward of the owner-sharded form: the gradient rows [row_lo, row_hi) this rank owns, from every triple that touches one of
 * them (as a user, a positive or a negative); x = <u,p> - <u,n> is recomputed from the gathered table (the rows are loaded for
 * the gradient anyway) and the norms are the global ones from hgr_bpr_l2_finish_f32.  d_rows zero-filled by the caller. */
int hgr_bpr_l2_bwd_owned_f32(const float *table, int64_t n_rows, int32_t D, const int64_t *u, const int64_t *p, const int64_t *n,
                             int64_t batch, float reg, float batch_size_div, const float *norms, const float *grad_out,
                             int64_t row_lo, int64_t row_hi, float *d_rows, hgr_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Full-ranking evaluation: GraphRecommender.test (base/graph_recommender.py:61-92, identical in
 * base/main_recommender.py:64-100) with predict (model/graph/LightGCN.py:99-102) and find_k_largest
 * (util/algorithm.py:143-173) fused: for every test user the scores against ALL items, the user's
 * training items replaced by -10e8 (they stay candidates, as in the reference), and the K best.
 *   user_emb [n_users, D], item_emb [n_items, D]   fp32 row-major
 *   test_users [n_test]                            dense user ids (int32)
 *   train_indptr [n_users + 1] (int64), train_indices (int32, ascending inside a row): the training
 *                                                  interaction matrix (Interaction.interaction_mat)
 *   out_ids [n_test, K] (int32), out_scores [n_test, K]: best first
 * Scores are DEFINED as the ascending-k fused multiply-add chain of fp32 products (the reference's BLAS
 * summation order is unspecified); out_scores holds exactly those values.
 * mode 0 ("exact"):    true top-K, score descending, ties by ascending item id, no duplicates.
 * mode 1 ("refquirk"): find_k_largest as shipped, which visits the first K candidates twice, so an item
 *                      with id < K that makes the list appears twice (SURVEY.md F9); K <= 256.
 * engine 0: tcgen05 tensor path when D == 64 and K <= 256 (candidate generation with 2 x bf16 split operands
 *           and a proven error bound, exact fp32 re-scoring of the candidates; results identical to
 *           engine 1), else SIMT.
 * engine 1: SIMT fp32 brute force (any K <= n_items in mode 0).
 * engine 2: tensor path (D == 64 and K <= 256) or HGR_ERR_INVALID.
 * stats (device uint64[4], optional, caller zeroes): candidates emitted by the tensor stage, candidates
 * re-scored, users that overflowed to the brute-force fallback, and the largest observed
 * |tensor score - fp32 score| in parts per million of the proven error bound (always < 1e6).
 * ------------------------------------------------------------------------------------------- */
size_t hgr_fullrank_topk_workspace_bytes(int64_t n_test, int64_t n_items, int32_t D, int32_t K, int32_t engine);
int hgr_fullrank_topk_f32(const float *user_emb, int64_t n_users, const float *item_emb, int64_t n_items, int32_t D,
                          const int32_t *test_users, int64_t n_test, const int64_t *train_indptr,
                          const int32_t *train_indices, int32_t K, int32_t mode, int32_t engine, int32_t *out_ids,
                          float *out_scores, uint64_t *stats, void *workspace, size_t workspace_bytes,
                          hgr_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Contrastive (SSL) losses fused with their gathers and row normalisation (util/loss_torch.py).
 *   kind 0  contrastLoss(embeds1, embeds2, nodes, temp)   util/loss_torch.py:103-110 (HCCF.py:62-66, HGNN_HD3.py:345-350)
 *   kind 1  InfoNCE(view1, view2, temperature, b_cos)     util/loss_torch.py:32-40   (SGL.py:167-180)
 * E1 [n_rows1, D], E2 [n_rows2, D]; nodes int64 [M] picks the rows (NULL: rows 0..M-1 of both tables, the InfoNCE
 * call shape).  A repeated id gives duplicate rows and columns of the logits, and its table row receives the sum of
 * the gradients of its copies (the reference passes torch.unique(...)).  normalize = F.normalize of the rows
 * (always on for kind 0, b_cos for kind 1).  loss: device float[1].  `saved` (hgr_ssl_workspace_bytes(M, D), 256-byte
 * aligned) carries the normalised rows, row sums and coefficients to the backward call.  The [M, M] logits are never
 * materialised.  Backward: dE1 / dE2 ([n_rows, D], zero-filled by the caller; either may be NULL for a detached
 * operand) receive grad_out[0] * d loss / d E at the picked rows.  A NEGATIVE entry of nodes is an inactive slot: it
 * takes no part in the loss (no row, no column, not counted in the mean), which lets a fixed-size batch stand in for
 * torch.unique's variable-length result (sorted ids with the repeats replaced by -1: CUDA-graph capturable).  Entries
 * beyond the tables are counted in *bad_index_count (device int, caller zeroes) and skipped the same way.
 * ------------------------------------------------------------------------------------------- */
size_t hgr_ssl_workspace_bytes(int64_t M, int32_t D);
int hgr_ssl_loss_fwd_f32(const float *E1, const float *E2, int64_t n_rows1, int64_t n_rows2, int32_t D, const int64_t *nodes,
                         int64_t M, float temp, int32_t kind, int32_t normalize, float *loss, void *saved, size_t saved_bytes,
                         int32_t *bad_index_count, hgr_stream_t stream);
int hgr_ssl_loss_bwd_f32(int64_t n_rows1, int64_t n_rows2, int32_t D, const int64_t *nodes, int64_t M, float temp, int32_t normalize,
                         void *saved, size_t saved_bytes, const float *grad_out, float *dE1, float *dE2, hgr_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * BPR negative sampling on the device: the body of next_batch_pairwise (util/sampler.py:237-264).
 * Positives of the batch are training pairs perm[perm_offset .. perm_offset + batch) of (edge_u, edge_i)
 * (perm == NULL: the pairs themselves in stored order); for each, n_negs items drawn uniformly from
 * [0, n_items) and re-drawn while they are in the user's training row (train_indptr / train_indices, columns
 * ascending).  out_u, out_p: int64 [batch]; out_n: int64 [batch * n_negs] (the reference's j_idx order).
 * Philox4x32-10(seed) with counter (stream_offset + sample index, attempt): reproducible, independent of the
 * launch geometry; pass a different stream_offset (e.g. the number of samples drawn so far) for every batch.
 * *gave_up (device int, optional, caller zeroes) counts samples still colliding after 256 draws.
 * ------------------------------------------------------------------------------------------- */
int hgr_bpr_sample(const int32_t *edge_u, const int32_t *edge_i, int64_t n_edges, const int64_t *perm, int64_t perm_offset,
                   int64_t batch, int32_t n_negs, const int64_t *train_indptr, const int32_t *train_indices, int32_t n_items,
                   uint64_t seed, uint64_t stream_offset, int64_t *out_u, int64_t *out_p, int64_t *out_n, int32_t *gave_up,
                   hgr_stream_t stream);

/* Per-user pieces of the ranking metrics (util/evaluation.py: Metric.hits :9-15, Metric.NDCG :85-97) from the id matrix of
 * hgr_fullrank_topk_f32: for every test user r and every N = top_n[q] (ascending, q < n_top <= 16)
 *   hits[r][q] = | set(truth items of r) & set(ids[r][:N]) |,   dcg[r][q] = sum of disc[p] over hit positions p < N
 * (double, position order; disc[p] = 1 / math.log(p + 2, 2) supplied by the host).  truth rows (truth_indptr int64
 * [n_test + 1], truth_items int32) must be sorted ascending; -1 entries (items unseen in training) never match.
 * The sums over users are left to the host so that the rounded strings equal the reference's. */
int hgr_rank_metrics(const int32_t *ids, int64_t n_test, int32_t K, const int64_t *truth_indptr, const int32_t *truth_items,
                     const int32_t *top_n, int32_t n_top, const double *disc, int32_t *hits, double *dcg, hgr_stream_t stream);

/* The sums over test users that turn those per-user pieces into the metric values (util/evaluation.py: Metric.hit_ratio :18-30,
 * precision :45-48, recall :50-53, NDCG :85-97), accumulated on the device in the reference's own order of additions:
 *   hit_sum[q]    = sum_r hits[r][q]                                  (integers)
 *   recall_sum[q] = sum_r hits[r][q] / n_truth(r)                     (python's builtin sum(): `compensated` != 0 selects the
 *                                                                      Neumaier summation of python >= 3.12, 0 the plain one)
 *   ndcg_sum[q]   = sum_r dcg[r][q] / idcg_tab[min(n_truth(r), N_q)]  (plain sequential `+=`, users in row order)
 * idcg_tab[k] = sum_{p<k} 1 / math.log(p + 2, 2), accumulated by the host in python doubles (idcg_len entries).
 * One thread per sum walks the users in order (the order IS the result); the per-user terms are formed in parallel. */
int hgr_rank_metric_sums(const int32_t *hits, const double *dcg, const int64_t *truth_indptr, int64_t n_test, int32_t n_top,
                         const int32_t *top_n, const double *idcg_tab, int32_t idcg_len, int32_t compensated, int64_t *hit_sum,
                         double *recall_sum, double *ndcg_sum, hgr_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* HGR_H_ */
