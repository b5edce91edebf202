/*
 * xpgnn_b200.h -- C ABI of the B200-native perturbation engine (libxpgnn_b200.so).
 *
 * Drop-in boundary for the perturbation hot path of `pathway_explanations`
 * (reference: andres2631996/bikg_graph_explainability_public).  Every entry point cites the
 * reference interface it replaces (file:line relative to the reference root).  The reference
 * is pure Python, so its "FFI" is a ctypes binding (see INTEGRATION.md); nothing in these
 * signatures is a torch type.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in `_host`;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, no call
 *     synchronises unless its comment says so;
 *   - return value 0 = success, anything else = failure, text via xpgnn_last_error();
 *   - node ids are int32 in engine structures (N, E < 2^31), int64 at the reference-facing
 *     k-hop boundary (PyG edge_index is int64);
 *   - coalition bits are packed node-major: act[v * W + w] bit b  <=>  node v is active in
 *     coalition (32*w + b).  W = ceil(S / 32).  A "tile" is one such 32-coalition word.
 */
#ifndef XPGNN_B200_H
#define XPGNN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XPGNN_ABI_VERSION 1

const char* xpgnn_last_error(void);
int xpgnn_abi_version(void);
/* number of kernel launches issued by this library since load (bench.py `gpu_launches`) */
int64_t xpgnn_launch_count(void);

/* Engine options.  Every option selects between implementations of the same function (kernel variant, occupancy, path
 * selection); none changes what is computed beyond floating-point summation order.  The XPGNN_<NAME> environment
 * variables only seed the defaults and are read ONCE, at the first use of the library; afterwards an option changes
 * only through this call.  Names (csrc/knobs.cuh): compact, compact_hetero, cw, l0_lists, occ, seg, seg_occ, seg_skew, seg_tma,
 * seg_pf, seg_carve, l2_stream, l2_gather, sched_static, long_rows, l0_slices, occ16, l0_multi, l1_multi, l0_ws, l0_wait_ns,
 * dense_wait_ns, dense_tma (0: register loaders instead of TMA gather4 for the A operand of the layer >= 1 TF32x3 transforms;
 * bit-identical), dense_simt (1: exact fp32 FMA transforms instead of the 3xTF32 tensor-core products of the fp32 plan),
 * prune_l0, fused, fused_sb.
 * The reference has no counterpart (its arch call is a black box, model.py:104-112). */
int xpgnn_set_option(const char* name, int32_t value);
int xpgnn_get_option(const char* name, int32_t* value);

/* ------------------------------------------------------------------------------------------
 * a1/a4  RNG stream + coalition masks
 * replaces: torch CPU generator draws inside Mask.mask_generator (masks.py:262-397),
 *           get_internal_mask (masks.py:80-136), get_external_indices (masks.py:138-194),
 *           Pathways.mask_generator / activate_dead_mask / pathway_mask2node_mask
 *           (pathways.py:234-385), shapley_mask (masks.py:231-260), torch.randperm (masks.py:385)
 * ---------------------------------------------------------------------------------------- */

/* Replays at::mt19937.  state624: 624 words in/out; pos: in/out scalar (0..624, 624 = twist
 * before the next output).  Writes n tempered 32-bit outputs to draws. */
int xpgnn_mt19937_draw(uint32_t* state624, int32_t* pos, uint32_t* draws, int64_t n, void* stream);

/* Host-computed row plan of the mask generator (one entry per community *position*, i.e. after
 * the descending-length argsort of masks.py:314). */
typedef struct {
  int32_t n_elements;         /* N_sub (mask columns)                                     */
  int32_t n_communities;      /* C                                                        */
  int32_t n_positions;        /* communities actually visited (masks.py:344-346 break)     */
  int32_t n_rows;             /* sum of size[] over positions                              */
  const int32_t* com_ptr;     /* [C+1]  member ranges, community order = caller's list     */
  const int32_t* com_idx;     /* [com_ptr[C]] member node ids, ascending inside community  */
  const int32_t* node_ptr;    /* [N+1]  inverse map: memberships of each node              */
  const int32_t* node_com;    /* [..]   community id of each membership                    */
  const int32_t* node_slot;   /* [..]   rank of the node inside that (sorted) community    */
  const int32_t* order;       /* [n_positions] community id at each position               */
  const int32_t* size;        /* [n_positions] rows of the block (masks.py:117,125)        */
  const int32_t* size_int;    /* [n_positions] internal-only rows (masks.py:120,124)       */
  const int32_t* row_start;   /* [n_positions+1] first pre-shuffle row of each block       */
} xpgnn_mask_plan_t;

/* Upper bound of the draws the plan can consume (incl. dead-mask repairs and the shuffle). */
int64_t xpgnn_mask_max_draws(const int32_t* size_host, const int32_t* size_int_host,
                             const int32_t* len_host, int32_t n_positions, int32_t n_communities,
                             int32_t shuffle);

/* Walks the blocks in stream order and resolves the data-dependent stream offsets (dead-mask
 * repair, pathways.py:285-334).  offsets: [n_positions*4] = {internal, external, odd row or -1,
 * repaired community or -1}; consumed[0] = draws used before the shuffle.
 * If shuffle != 0 also runs torch.randperm(n_rows) (Fisher-Yates, masks.py:385) into ind and adds
 * its n_rows-1 draws to consumed[0]. */
int xpgnn_mask_resolve(const xpgnn_mask_plan_t* plan_host, const uint32_t* draws, int64_t* offsets,
                       int64_t* consumed, int32_t shuffle, int32_t* ind, void* stream);

/* Expands coalitions [0, n_out) of the shuffled order (row s = pre-shuffle row ind[s]).
 * Any of the outputs may be NULL.  mask_rowmajor: uint8 [n_out][N] (the reference's bool matrix);
 * act: packed node-major [N][W]; pathway_rows: int32 [n_out]; popcount: int32 [n_out]. */
int xpgnn_mask_expand(const xpgnn_mask_plan_t* plan_host, const uint32_t* draws,
                      const int64_t* offsets, const int32_t* ind, int32_t n_out, uint8_t* mask_rowmajor,
                      uint32_t* act, int32_t W, int32_t* pathway_rows, int32_t* popcount, void* stream);

/* Shapley mode (masks.py:231-260): bit (r, v) = draws[r * N + v] & 1, rows permuted by ind. */
int xpgnn_shapley_expand(const uint32_t* draws, const int32_t* ind, int32_t n_out, int32_t n_elements,
                         uint8_t* mask_rowmajor, uint32_t* act, int32_t W, int32_t* popcount,
                         void* stream);

/* torch.randperm(n) from the stream: consumes n-1 draws (single CTA). */
int xpgnn_randperm(const uint32_t* draws, int32_t n, int32_t* perm, void* stream);

/* Row-major uint8 mask [S][N] -> packed node-major act [N][W] and popcounts (used when the
 * caller brings its own masks, e.g. the synthetic throughput workload). */
int xpgnn_pack_mask(const uint8_t* mask_rowmajor, int32_t S, int32_t N, uint32_t* act, int32_t W,
                    int32_t* popcount, void* stream);

/* ------------------------------------------------------------------------------------------
 * a2  k-hop computational graph
 * replaces: Data.comp_graph (data.py:281-361) -> torch_geometric.utils.k_hop_subgraph
 * ---------------------------------------------------------------------------------------- */

/* edge_index: int64 [2][E] (row 0 = source, row 1 = target).  Frontier BFS over in-edges for
 * `hops` levels from `query`, then the induced subgraph.  Outputs (all sized by the caller for the
 * worst case): subset int64 [N] ascending node ids; relabel int32 [N] (-1 outside);
 * hop int8 [N] first level a node was reached at (-1 outside); edge_mask uint8 [E];
 * sub_edge_index int64 [2][E] with row stride E (first counts[1] columns valid, original order,
 * relabelled); counts int64 [3] = {N_sub, E_sub, number of edges with an endpoint outside [0, N)}.  Such edges are
 * ignored by the kernels and the caller raises (PyG raises an index error); N and E must fit int32.  If no edge
 * survives, one self loop on the query is emitted (data.py:337-339) and counts[1] = 1. */
int xpgnn_khop_subgraph(const int64_t* edge_index, int64_t E, int64_t N, int64_t query, int32_t hops,
                        int64_t* subset, int32_t* relabel, int8_t* hop, uint8_t* edge_mask,
                        int64_t* sub_edge_index, int64_t* counts, void* stream);

/* CSR by destination.  src/dst int64 [E].  Keeps edge order inside a row (stable).  If
 * drop_self_loops, edges with src == dst are removed (GCN's add_remaining_self_loops replaces
 * them by one unit loop that the engine adds analytically).  rowptr int32 [N+1], col int32 [E],
 * n_kept int64 [1]. */
int xpgnn_build_csr(const int64_t* src, const int64_t* dst, int64_t E, int64_t N, int32_t drop_self_loops,
                    int32_t* rowptr, int32_t* col, int64_t* n_kept, void* stream);

/* Multi-query k-hop: the computational graphs of Q <= 64 queries (repeats allowed) in the passes one
 * query needs.  One uint64 reach word per node and level (bit q = reached from queries[q] at that
 * level, PyG's re-expansion of the whole previous level), so the workspace is
 * xpgnn_khop_multi_workspace_bytes(N, hops) = 8 N (hops + 1) plus a few KB, independent of E and Q.
 * Two calls share the caller-held workspace:
 *   count: counts int64 [2Q + 1] = {N_q for every q, E_q for every q (before the self-loop rule),
 *          number of edges with an endpoint outside [0, N)};
 *   emit:  node_off / edge_off int64 [Q + 1] are the caller's exclusive prefix sums of N_q and of
 *          max(E_q, 1), in device memory; the union is written block by block:
 *          subset int64 [node_off[Q]] (each query's node ids ascending), level int8 [node_off[Q]]
 *          (first level the node was reached at from its query), sub_ind int64 [Q] (rank of the query
 *          inside its own block), sub_edge_index int64 [2][edge_off[Q]] (row stride edge_off[Q]; each
 *          query's induced edges in original order, relabelled to union positions, i.e. node_off[q]
 *          added) and edge_id int64 [edge_off[Q]] (optional: the input column of each union edge).
 *          A query with no induced edge gets one self loop on itself (edge_id -1), as
 *          xpgnn_khop_subgraph does.  Every block equals what xpgnn_khop_subgraph gives for that query. */
int64_t xpgnn_khop_multi_workspace_bytes(int64_t N, int32_t hops);
int xpgnn_khop_multi_count(const int64_t* edge_index, int64_t E, int64_t N, const int64_t* queries, int32_t Q,
                           int32_t hops, void* workspace, int64_t workspace_bytes, int64_t* counts, void* stream);
int xpgnn_khop_multi_emit(const int64_t* edge_index, int64_t E, int64_t N, const int64_t* queries, int32_t Q,
                          int32_t hops, const void* workspace, int64_t workspace_bytes, const int64_t* counts,
                          const int64_t* node_off, const int64_t* edge_off, int64_t n_union_edges, int64_t* subset,
                          int8_t* level, int64_t* sub_ind, int64_t* sub_edge_index, int64_t* edge_id, void* stream);

/* ------------------------------------------------------------------------------------------
 * a5/a6/a7  coalition-batched masked message passing
 * replaces: Data.perturbator / build_edge_mask / perturb_node / concat_features
 *           (data.py:390-648), Model.infer / predict_hetero_output / extract_node_edge_output
 *           (model.py:62-328) and the PyG GCNConv / SAGEConv / HeteroConv forward they call.
 * Nothing is materialised: edge (u->v) is active in coalition s iff both endpoint bits are set.
 * ---------------------------------------------------------------------------------------- */

enum { XPGNN_CONV_GCN = 0, XPGNN_CONV_SAGE_MEAN = 1 };
enum { XPGNN_ACT_NONE = 0, XPGNN_ACT_RELU = 1, XPGNN_ACT_SIGMOID = 2 };

typedef struct {
  int32_t conv_kind;
  int32_t src_lo, src_hi;     /* flattened id range of the source node type                 */
  int32_t dst_lo, dst_hi;     /* flattened id range of the destination node type            */
  int32_t n_edges;            /* entries of col (after self-loop removal for GCN)            */
  const int32_t* rowptr;      /* [N+1] in-edges by flattened destination id                  */
  const int32_t* col;         /* [E_r] flattened source ids (GCN: self loops already dropped) */
  const float* w_nbr;         /* [h_out][h_in]  GCN lin.weight | SAGE lin_l.weight            */
  const float* b_nbr;         /* [h_out] or NULL  GCN bias | SAGE lin_l.bias                  */
  const float* w_root;        /* [h_out][h_in]  SAGE lin_r.weight, NULL for GCN               */
} xpgnn_relation_t;

typedef struct {
  int32_t n_rel;
  const xpgnn_relation_t* rel_host; /* host array */
  int32_t h_in, h_out;
  int32_t act;                /* activation applied to the layer output                       */
} xpgnn_layer_t;

typedef struct {
  int32_t in, out, act;
  const float* w;             /* [out][in] */
  const float* b;             /* [out] or NULL */
} xpgnn_dense_t;

typedef struct {
  int32_t n_nodes;            /* flattened node count N                                       */
  int32_t f_in;               /* (padded) input feature width                                 */
  const float* x;             /* [N][f_in]                                                    */
  int32_t n_layers;
  const xpgnn_layer_t* layers_host;
  int32_t n_head;
  const xpgnn_dense_t* head_host;
  int32_t n_query;
  const int32_t* query;       /* [n_query] flattened node ids whose prediction is read        */
  int32_t out_col;            /* column of the head output that is read (reference: 0)        */
  int32_t prune;              /* 0: every conv layer on every row (reference-equivalent work)
                                 1: only rows whose value can reach a query                  */
  const int8_t* hop;          /* [N] BFS level from the queries (needed when prune = 1)        */
  int32_t zero_edge_rule;     /* 1: a coalition with no active edge yields 0 (model.py:213-215) */
  int32_t precision;          /* 0: fp32 storage, transforms as 3xTF32 tcgen05 MMAs (1e-4 bar);
                                 1: fp32 storage, bf16 tcgen05 transforms (2e-2 bar);
                                 2: bf16 transforms + bf16 storage of the per-coalition activations where the
                                    compact path supports it (GCN stacks, widths % 64 == 0), else as 1 */
} xpgnn_plan_t;

/* Bytes of scratch xpgnn_forward needs to process `tile_coalitions` (1..32, power of two)
 * coalitions at a time.  xpgnn_forward picks the largest tile that fits the workspace it is given. */
int64_t xpgnn_forward_workspace_bytes(const xpgnn_plan_t* plan_host, int32_t tile_coalitions);

/* Evaluates coalitions [s0, s0 + n_s) (s0 % 32 == 0).  y: float [n_s][n_query] (row stride
 * n_query), y[s - s0][q] = head(conv stack)(query q) under coalition s.
 * stats (optional, int64 [4], accumulated): {edge visits, active edge visits, spmm launches, tiles}. */
int xpgnn_forward(const xpgnn_plan_t* plan_host, const uint32_t* act, int32_t W, int32_t s0, int32_t n_s,
                  float* y, void* workspace, int64_t workspace_bytes, int64_t* stats, void* stream);

/* Dense row transform out = act(in * w^T + b) (the coalition-invariant X*W of the first layer and
 * the per-layer transforms); exposed for tests and for the unperturbed forward of the layers. */
int xpgnn_dense_rows(const float* in, int64_t rows, int32_t k, int32_t ld_in, const float* w, const float* b,
                     int32_t n_out, int32_t act, float* out, int32_t ld_out, int32_t accumulate,
                     int32_t precision, void* stream);

/* Measurement hook (bench.py roofline): when enabled, every engine kernel launch is bracketed by
 * CUDA events on its stream.  xpgnn_profile_read synchronises those events and returns, per
 * category {masked degree, SpMM on the coalition-invariant operand (layer 0), SpMM on coalition-
 * specific activations (layers >= 1), dense transform, head, per-tile compaction of the active edge lists},
 * the summed device time in ms and the number of launches.  Both arrays are HOST arrays of 6 entries. */
int xpgnn_profile(int32_t enable);
int xpgnn_profile_read(double* ms_host, int64_t* launches_host);

/* ------------------------------------------------------------------------------------------
 * a8  SHAP kernel weights
 * replaces: Kernel.compute / original_shap_kernel / approximate_shap_kernel (kernels.py:22-174)
 * ---------------------------------------------------------------------------------------- */

/* popcount int32 [S]; M = mask columns.  Exact branch (M-1 <= 1000): table = binom(M, j),
 * j = 0..M (M+1 doubles), n_tables = 1.  Approx branch: tables are binom(ref_i, j), j < ref_i for
 * ref_0 = 1000, ref_{i+1} = int(0.9 ref_i) ... concatenated; table_ptr int32 [n_tables+1].
 * The shrink loop of kernels.py:154-162 runs per batch of `batch` consecutive coalitions.
 * out: double [S]. */
int xpgnn_shap_weights(const int32_t* popcount, int32_t S, int32_t M, int32_t batch, const double* tables,
                       const int32_t* table_ptr, int32_t n_tables, double* out, void* stream);

/* ------------------------------------------------------------------------------------------
 * a9  weighted linear surrogate (one Adam step per batch, in batch order)
 * replaces: train_model / LinearRegression / regularizer / weighted_mse_loss /
 *           optimizer_scheduler (wlm.py:17-278, 441-520)
 * ---------------------------------------------------------------------------------------- */

/* act [N][W] packed; y float [S] (query prediction per coalition); kern double [S]; w float [N]
 * in: initial weights, out: fitted weights.  broadcast_y = 1 reproduces the (B,1)-target
 * broadcast of wlm.py:517.  losses (optional) double [ceil(S / batch)]. */
int xpgnn_wlm_fit(const uint32_t* act, int32_t W, int32_t N, int32_t S, int32_t batch, const float* y,
                  const double* kern, float* w, double lr, double l1_lambda, double weight_decay,
                  int32_t broadcast_y, double* losses, void* stream);

/* One surrogate of xpgnn_wlm_fit_batch: its coalition bits start at act[act_off] (row stride W of the
 * call), its predictions at y[y_off] (row stride ldy of the call), its kernel weights at kern[kern_off],
 * its weights at w[w_off] (N entries, initial in, fitted out); losses (optional) double [ceil(S / batch)]. */
typedef struct {
  int64_t act_off, y_off, kern_off, w_off;
  int32_t n, s, batch, pad_;
  double* losses;
} xpgnn_fit_query_t;

/* Q independent xpgnn_wlm_fit problems in one launch sequence: three launches per step index for the
 * whole batch; a surrogate with fewer steps drops out of later launches.  Every surrogate's weights
 * and losses are bit-identical to xpgnn_wlm_fit on the same inputs.  The hyper-parameters and
 * broadcast_y are shared. */
int xpgnn_wlm_fit_batch(const uint32_t* act, int32_t W, const float* y, int64_t ldy, const double* kern, float* w,
                        const xpgnn_fit_query_t* queries_host, int32_t Q, double lr, double l1_lambda,
                        double weight_decay, int32_t broadcast_y, void* stream);

/* ------------------------------------------------------------------------------------------
 * a10  aggregation
 * replaces: Explainer.weight_stacking (explainer.py:288-314), Pathways.aggregate (pathways.py:387-429)
 * ---------------------------------------------------------------------------------------- */

/* weights float [times][N] -> mean, population std float [N]. */
int xpgnn_repeat_stats(const float* weights, int32_t times, int32_t N, float* mean, float* std, void* stream);

/* score[c] = mean(w[com_idx[com_ptr[c] .. com_ptr[c+1])]) (NaN for an empty community). */
int xpgnn_community_mean(const float* w, const int32_t* com_ptr, const int32_t* com_idx, int32_t C,
                         float* score, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* XPGNN_B200_H */
