/*
 * qot_b200.h -- C ABI of libqot_b200.so: the B200 (sm_100a) kernels behind the
 * message-passing hot path of santiagolmedo/gnn_qot_estimation.
 *
 * The reference has no FFI: its "plugin API" for this path is the Python
 * nn.Module contract of TopologicalGNN (topological_training/models.py:6-64) and
 * LightpathGNN (lightpath_training/models.py:7-45), whose arithmetic lives in
 * PyTorch Geometric layers.  Each entry point below replaces the PyG call named
 * in its comment; gnn_qot_estimation_b200/ binds them with ctypes and keeps the
 * reference's module names/constructors/forward(data) on top (INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host;
 *   - the caller owns every buffer (inputs, outputs, workspace); the library never
 *     allocates, frees or retains memory;
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); no entry
 *     point synchronises, so every call is CUDA-graph capturable;
 *   - return value: 0 = ok, <0 = QOT_E_* ; qot_last_error() gives a thread-local
 *     message for the most recent failure on the calling thread;
 *   - features are fp32, API indices int64 (as the reference tensors are), internal
 *     CSR indices int32;
 *   - results are deterministic: segments are sorted, reductions have a fixed
 *     order, no floating-point atomics anywhere.
 */
#ifndef QOT_B200_H_
#define QOT_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QOT_OK 0
#define QOT_E_BADARG (-1)      /* null pointer / negative size / unsupported shape */
#define QOT_E_WORKSPACE (-2)   /* workspace too small */
#define QOT_E_CUDA (-3)        /* a CUDA runtime call or launch failed */

#define QOT_EDGE_DIM 4         /* edge_attr width (topological_training/train.py:52) */
#define QOT_EDGE_HID 8         /* edge-MLP hidden = 2*edge_dim (models.py:21)        */
#define QOT_GAT_IN 5           /* lightpath node features (lightpath dataset.py:45)  */
#define QOT_GAT_HEADS 4        /* lightpath_training/models.py:13                    */
#define QOT_GAT_C 32           /* hidden_channels per head (train.py:52)             */
#define QOT_GAT_HC 128         /* heads * C                                          */
#define QOT_OUT 3              /* osnr, snr, ber                                     */

const char* qot_last_error(void);
int qot_version(void);

/* ------------------------------------------------------------------------ */
/* (1) collate + CSR: replaces torch_geometric.loader.DataLoader's            */
/*     Batch.from_data_list (topological_training/train.py:93-95,             */
/*     lightpath_training/train.py:94-96) and the scatter-by-index inside     */
/*     PyG's MessagePassing.propagate.                                        */
/* ------------------------------------------------------------------------ */

/* A packed graph store (all graphs of a dataset, flat arrays in HBM). */
typedef struct {
  const int64_t* node_ptr;   /* [G+1] node offsets                              */
  const int64_t* edge_ptr;   /* [G+1] directed-edge offsets                     */
  const int32_t* edge_src;   /* [E_tot] graph-local source id                   */
  const int32_t* edge_dst;   /* [E_tot] graph-local target id                   */
  const float* node_feat;    /* [N_tot, node_dim] or NULL (topological: x=None) */
  const float* edge_feat;    /* [E_tot, edge_dim] or NULL (lightpath)           */
  const float* y;            /* [G, y_dim]                                      */
  int32_t node_dim, edge_dim, y_dim;
} qot_store_t;

/* Collate `B` graphs `graph_ids[b]` of the store into one batch.
 * out_ptr/out_eptr [B+1] int64 must already hold the batch-local node / edge
 * offsets (the host owns a copy of node_ptr/edge_ptr and computes them while
 * sizing the outputs -- no device->host sync).  Writes
 *   x [N,node_dim], edge_index [2,E] int64 (offset by the running node count),
 *   edge_attr [E,edge_dim], batch [N] int64, node_ids [N] int64 (0..n_g-1 per
 *   graph, topological_training/dataset.py:78), y [B,y_dim].
 * Any output pointer may be NULL to skip it. */
int qot_collate(const qot_store_t* store, const int64_t* graph_ids, int64_t B,
                const int64_t* out_ptr, const int64_t* out_eptr, int64_t N, int64_t E,
                float* x, int64_t* edge_index, float* edge_attr, int64_t* batch,
                int64_t* node_ids, float* y, void* stream);

/* Workspace for qot_build_csr. */
size_t qot_csr_workspace_bytes(int64_t N, int64_t E);

/* Group the E edges of edge_index [2,E] (int64) by row `by` (1 = by destination,
 * the forward CSR; 0 = by source, the transposed CSR the backward kernels use),
 * STABLE in the original edge order.  flags: bit0 = drop self loops, bit1 = append
 * one self loop per node as the last entry of its row (GATConv's
 * remove_self_loops + add_self_loops; appended loops get eid = E + node).
 *   rowptr [N+1] int32, nbr [E'] int32 (the other endpoint), eid [E'] int32
 *   (original edge id), E' <= E + N.
 * status (optional, int32[1]) is set non-zero on device if an index is out of
 * range [0,N). */
int qot_build_csr(const int64_t* edge_index, int64_t E, int64_t N, int by, int flags,
                  int32_t* rowptr, int32_t* nbr, int32_t* eid, int32_t* status,
                  void* ws, size_t ws_bytes, void* stream);

/* gptr [B+1] int64 from a sorted `batch` [N] (== PyG Batch.ptr): gptr[g] = first
 * node whose graph id is >= g. */
int qot_graph_ptr(const int64_t* batch, int64_t N, int64_t B, int64_t* gptr, void* stream);

/* eptr [B+1] int64: first edge whose source node lies in a graph >= g.  Valid when
 * the edges of edge_index [2,E] are grouped by graph in ascending order (every
 * collate emits them so); status[0] (int32) is set non-zero otherwise, and also when an
 * endpoint lies outside [0,N) or an edge joins two different graphs -- the fused
 * inference kernel relies on this check for batches that do not come from a collate. */
int qot_edge_ptr(const int64_t* edge_index, int64_t E, const int64_t* batch, int64_t N,
                 int64_t B, int64_t* eptr, int32_t* status, void* stream);

/* ------------------------------------------------------------------------ */
/* dense node-wise projections (FP32-exact FFMA tiles)                        */
/* ------------------------------------------------------------------------ */

/* C[M,Nc] (ldc) = op(A)[M,K] * op(B)[K,Nc] (+ bias[Nc]) with arbitrary element
 * strides: A(m,k) = A[m*a_rs + k*a_cs], B(k,n) = B[k*b_rs + n*b_cs].
 * gather (optional int64 [M]): row m of A is read at row gather[m] (embedding
 * lookup, topological_training/models.py:52).  Replaces the addmm calls inside
 * TransformerConv / NNConv. */
int qot_gemm(const float* A, int64_t a_rs, int64_t a_cs, const int64_t* gather,
             const float* B, int64_t b_rs, int64_t b_cs, const float* bias,
             float* C, int64_t ldc, int64_t M, int64_t Nc, int64_t K, void* stream);

/* The same projection on the tensor cores (tcgen05.mma kind::tf32, TMEM accumulator) with
 * fp32-level accuracy: C[M,Nc] (ldc) = A[gather ? gather[m] : m, :K] (lda) * W[Nc,:K]^T (ldw)
 * (+ bias[Nc]), three TF32 products per k-step on hi/lo-split operands.  For hidden widths where
 * the projection is a real contraction (K % 32 == 0; BASELINE cfg 5, H = 256); lda, ldw multiples
 * of 4, 16-byte aligned bases.  status (optional, device int32[1]): bit 1 = a pipeline barrier
 * timed out (result undefined).  ws: room for the hi / lo halves of both operands, which a small
 * pre-pass writes once (it also performs the row gather). */
size_t qot_gemm_tf32x3_workspace_bytes(int64_t M, int64_t Nc, int64_t K);
/* Test hook, host only: the tile decomposition of a qot_gemm_tf32x3 / qot_wgrad_tf32x3 launch (pairs of tiles handed
 * to clusters of two CTAs).  out [rows][6] = m0, n0, first k-block, k-blocks, stores (0/1), split-K slice; returns the
 * number of rows, fills at most cap. */
int64_t qot_debug_gemm_tiles(int64_t M, int64_t Nc, int64_t K, int64_t kb_per_split, int64_t splits, int64_t* out,
                             int64_t cap);
int qot_gemm_tf32x3(const float* A, int64_t lda, const int64_t* gather, const float* W, int64_t ldw,
                    const float* bias, float* C, int64_t ldc, int64_t M, int64_t Nc, int64_t K,
                    int32_t* status, void* ws, size_t ws_bytes, void* stream);

/* Weight gradient on the tensor cores (same 3 x TF32 scheme): C[Mo,No] (ldc) = sum_r A[r,:Mo]^T
 * B[gather_b ? gather_b[r] : r, :No] over R rows.  Operands are transposed + split into K-major form,
 * the reduction is cut into split-K slices that are summed in a fixed order (deterministic). */
size_t qot_wgrad_tf32x3_workspace_bytes(int64_t R, int64_t Mo, int64_t No);
int qot_wgrad_tf32x3(const float* A, int64_t lda, const float* B, int64_t ldb, const int64_t* gather_b,
                     int64_t R, int64_t Mo, int64_t No, float* C, int64_t ldc, int32_t* status,
                     void* ws, size_t ws_bytes, void* stream);

/* Deterministic weight gradient: C[Mo,No] (ldc) = sum_r A[r,Mo]^T * B[r,No] over
 * R rows (row-major A [R,lda], B [R,ldb]); two-stage fixed-order reduction.
 * gather (optional int64 [R]) scatters by row: C[gather[r], :] += B[r, :] is NOT
 * supported here -- see qot_embedding_bwd. */
size_t qot_wgrad_workspace_bytes(int64_t R, int64_t Mo, int64_t No);
int qot_wgrad(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t R,
              int64_t Mo, int64_t No, float* C, int64_t ldc,
              void* ws, size_t ws_bytes, void* stream);

/* colsum[Nc] = sum_r A[r, :Nc]  (bias gradients), fixed order. */
size_t qot_colsum_workspace_bytes(int64_t R, int64_t Nc);
int qot_colsum(const float* A, int64_t lda, int64_t R, int64_t Nc, float* out,
               void* ws, size_t ws_bytes, void* stream);

/* out[r,:] = sum over p in [rowptr[r],rowptr[r+1]) of X[idx[p],:]  (H in 16/32/64/128/256;
 * `entries` = rowptr[R]).  Long rows are split over blocks and combined in a fixed order.
 * With the CSR of node_ids this is the deterministic embedding backward
 * (topological_training/models.py:52): dEmb[v] = sum of dX rows whose id is v. */
size_t qot_segment_sum_workspace_bytes(int64_t entries, int64_t R, int64_t H);
int qot_segment_sum(const float* X, const int32_t* rowptr, const int32_t* idx, int64_t entries,
                    int64_t R, int64_t H, float* out, void* ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------ */
/* (2) TransformerConv edge phase (topological_training/models.py:15-17,53)   */
/* ------------------------------------------------------------------------ */
/* qkvs [N,4H] = [q | k | v | skip] node projections (qot_gemm).  For each
 * destination row i of the CSR:  a_ij = q_i.(k_j + We a_ij)/sqrt(H);
 * alpha = softmax_i(a) (denominator + 1e-16);  out_i = sum alpha (v_j + We a_ij)
 * + skip_i;  then leaky_relu(slope) if slope != 1  (models.py:54).
 * Saves logit [E'] (CSR order), rmax [N], rden [N] for the backward when non-NULL. */
int qot_tconv_fwd(const float* qkvs, const int32_t* rowptr, const int32_t* src,
                  const int32_t* eid, const float* edge_attr, const float* We,
                  int64_t N, int64_t H, float slope, float* out, float* logit,
                  float* rmax, float* rden, void* stream);

/* Backward of qot_tconv_fwd.  dout [N,H] is the gradient w.r.t. the activated
 * output; `out` is the saved activated output (for the leaky_relu mask).
 * Produces dqkvs [N,4H] (gradient of the node projections) and dWe [H,4].
 * Needs the transposed CSR (t_rowptr/t_dst/t_eid from qot_build_csr(by=0)) and
 * pos_of_eid [E] (CSR slot of each original edge). */
size_t qot_tconv_bwd_workspace_bytes(int64_t N, int64_t E, int64_t H);
int qot_tconv_bwd(const float* qkvs, const int32_t* rowptr, const int32_t* src,
                  const int32_t* eid, const int32_t* t_rowptr, const int32_t* t_dst,
                  const int32_t* t_eid, const float* edge_attr, const float* We,
                  const float* out, const float* dout, const float* logit,
                  const float* rmax, const float* rden, int64_t N, int64_t E, int64_t H,
                  float slope, float* dqkvs, float* dWe,
                  void* ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------ */
/* (2) NNConv(aggr=mean) edge phase (topological_training/models.py:20-30,57) */
/* ------------------------------------------------------------------------ */
/* Factorised form (SURVEY.md Appendix A.2):  yr [N,(K+2)H], K = QOT_EDGE_HID:
 * slabs k<K: x P_k, slab K: x P_b (bias of the edge MLP's last layer), slab K+1:
 * x Wroot^T.  out_i = mean_j sum_k hh_e[k] yr[j,k,:] + yr[i,K+1,:] + bias, with
 * hh_e = [relu(W1 a_e + b1), 1]; then leaky_relu(slope). */
int qot_nnconv_fwd(const float* yr, const int32_t* rowptr, const int32_t* src,
                   const int32_t* eid, const float* edge_attr, const float* W1,
                   const float* b1, const float* bias, int64_t N, int64_t H, float slope,
                   float* out, void* stream);

/* Backward: dyr [N,(K+2)H], dW1 [K,4], db1 [K], dbias [H]. */
size_t qot_nnconv_bwd_workspace_bytes(int64_t N, int64_t E, int64_t H);
int qot_nnconv_bwd(const float* yr, const int32_t* rowptr, const int32_t* src,
                   const int32_t* eid, const int32_t* t_rowptr, const int32_t* t_dst,
                   const int32_t* t_eid, const float* edge_attr, const float* W1,
                   const float* b1, const float* out, const float* dout,
                   int64_t N, int64_t E, int64_t H, float slope,
                   float* dyr, float* dW1, float* db1, float* dbias,
                   void* ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------ */
/* (3) global_mean_pool + MLP head (topological_training/models.py:33-38,61-63) */
/* ------------------------------------------------------------------------ */
/* pooled [B,H] (saved for backward), hid [B,H] pre-activation (saved), out [B,3].
 * head: Linear(H,H) - LeakyReLU(0.01) - Linear(H,3). */
size_t qot_pool_mlp_fwd_workspace_bytes(int64_t N, int64_t B, int64_t H);
int qot_pool_mlp_fwd(const float* x, const int64_t* gptr, int64_t N, int64_t B, int64_t H,
                     const float* W1, const float* b1, const float* W2, const float* b2,
                     const float* hmask, float* pooled, float* hid, float* out,
                     void* ws, size_t ws_bytes, void* stream);

size_t qot_pool_mlp_bwd_workspace_bytes(int64_t B, int64_t H);
/* dx [N,H] (every node of graph g gets dpooled_g / n_g), dW1,db1,dW2,db2.
 * hmask (optional [B,H]) = dropout keep-mask/scale applied to the hidden
 * activation (NULL = none). */
int qot_pool_mlp_bwd(const float* dout, const float* pooled, const float* hid,
                     const float* hmask, const int64_t* gptr, int64_t N, int64_t B, int64_t H,
                     const float* W1, const float* W2, float* dx,
                     float* dW1, float* db1, float* dW2, float* db2,
                     void* ws, size_t ws_bytes, void* stream);

/* global_mean_pool on its own (PyG layer, topological_training/models.py:61 when the reference's
 * models.py is kept and only its layer imports are swapped): pooled [B,H]; backward
 * dx[n,:] = dpooled[graph(n),:] / n_graph.  ws: qot_mean_pool_workspace_bytes. */
size_t qot_mean_pool_workspace_bytes(int64_t N, int64_t B, int64_t H);
int qot_mean_pool_fwd(const float* x, const int64_t* gptr, int64_t N, int64_t B, int64_t H,
                      float* pooled, void* ws, size_t ws_bytes, void* stream);
int qot_mean_pool_bwd(const float* dpooled, const int64_t* gptr, int64_t N, int64_t B, int64_t H,
                      float* dx, void* ws, size_t ws_bytes, void* stream);

/* Fused SmoothL1Loss (mean reduction, beta) forward + gradient + running regression metrics:
 * replaces criterion(out, y) / loss.backward() entry / loss.item() / the per-batch .cpu() copies
 * for R^2 of topological_training/train.py:114-129 and lightpath_training/train.py:122-136.
 * pred [n,3]; target rows taken at target_rows[r] (NULL = r; y[lut_batch] without a gather).
 * loss [1] (optional), dpred [n,3] = d loss / d pred (optional), metrics [3,5] fp64 (optional):
 * per output column [count, sum y, sum y^2, sum (y-pred)^2, sum loss elements], ACCUMULATED. */
size_t qot_smooth_l1_workspace_bytes(int64_t n);
int qot_smooth_l1(const float* pred, const float* target, const int64_t* target_rows, int64_t n,
                  float beta, float* loss, float* dpred, double* metrics, void* ws, size_t ws_bytes,
                  void* stream);

/* ------------------------------------------------------------------------ */
/* LightpathGNN (lightpath_training/models.py:7-45)                           */
/* ------------------------------------------------------------------------ */
typedef struct {
  const float* lin_w;      /* conv1.lin.weight [128,5]        */
  const float* att_src;    /* conv1.att_src    [4,32]         */
  const float* att_dst;    /* conv1.att_dst    [4,32]         */
  const float* conv_bias;  /* conv1.bias       [128]          */
  const float* bn_w;       /* norm1.module.weight [128]       */
  const float* bn_b;       /* norm1.module.bias   [128]       */
  const float* bn_mean;    /* running_mean [128]              */
  const float* bn_var;     /* running_var  [128]              */
  const float* mlp_w1;     /* mlp.0.weight [32,128]           */
  const float* mlp_b1;     /* mlp.0.bias   [32]               */
  const float* mlp_w2;     /* mlp.3.weight [3,32]             */
  const float* mlp_b2;     /* mlp.3.bias   [3]                */
  float bn_eps;            /* 1e-5                            */
  int32_t is_lut_index;    /* column of x holding the LUT flag */
} qot_lightpath_params_t;

/* Fused eval-mode forward: GATConv -> BatchNorm(running stats) -> ReLU -> LUT
 * readout -> MLP (lightpath_training/models.py:26-45 under model.eval()), entry point
 * qot_lightpath_infer_stream below.  Graph-parallel, no cross-block dependency: graph g owns nodes
 * [gptr[g],gptr[g+1]) and edges [eptr[g],eptr[g+1]) of edge_index (as every collate produces
 * them; both endpoints of an edge lie in the graph that owns it), and its readout rows go to
 * [lut_ptr[g],lut_ptr[g+1]) -- lut_ptr [B+1] int64 is the exclusive prefix of the per-graph
 * count of LUT nodes (x[:,is_lut_index] == 1.0), an index array like gptr that the collate
 * builds once per batch (qot_lightpath_lut_ptr, or on the host).  Only the rows the readout
 * keeps are evaluated -- same values as computing all rows and selecting.  Outputs, in
 * ascending node order:
 *   out [L,3], lut_batch [L] int64 (graph id), lut_node [L] int32, n_lut[0] = L = lut_ptr[B].
 * status (int32[1], zeroed by the caller): bit 0 is set when lut_ptr does not describe x (a
 * graph holds a different number of LUT nodes); rows of such a graph are not written. */
size_t qot_lightpath_lut_ptr_workspace_bytes(int64_t B);
int qot_lightpath_lut_ptr(const float* x, const int64_t* gptr, int64_t N, int64_t B,
                          int32_t is_lut_index, int64_t* lut_ptr, void* ws, size_t ws_bytes,
                          void* stream);
/* Folds the parameters once per weight update (attention vectors through lin_w,
 * conv bias + BatchNorm running stats into one scale/shift, transposed MLP) into
 * `prepared` (qot_lightpath_prepared_floats() floats, 16-byte aligned). */
size_t qot_lightpath_prepared_floats(void);
int qot_lightpath_prepare(const qot_lightpath_params_t* p, float* prepared, void* stream);
/* Bytes of the z scratch a batch descriptor needs (20 floats per readout row, rows <= N); only the
 * QOT_LP_SPLIT_HEAD build of the kernel writes it. */
size_t qot_lightpath_infer_workspace_bytes(int64_t N);

/* The same forward over MANY batches in ONE launch of a persistent, warp-specialised kernel
 * (lp_stream_kernel, csrc/lightpath_stream.cu): the streaming form of the evaluation loop
 * lightpath_training/test.py:77-94 for batches already resident in HBM.  A batch is described by a
 * qot_lp_batch_t (reference layout, every pointer a device pointer); the caller keeps an array of them
 * in DEVICE memory, 16-byte aligned.  Work is cut into tiles of 16 consecutive graphs; tile0 of descriptor b is the number
 * of tiles before it (tile0[0] = 0, tile0[b+1] = tile0[b] + qot_lightpath_stream_tiles(B_b)).
 *   z       per-batch scratch of at least 20 floats per readout row (qot_lightpath_infer_workspace_bytes(N));
 *   status  one int32 per batch, ZERO on entry (pool them and clear the pool with one memset);
 *           bit 0: lut_ptr does not describe x, bit 2: a pipeline barrier timed out.
 * uniform_tiles: tiles per batch when every batch but the last has the same count, else 0 (the kernel
 * then searches tile0).  max_rows: an upper bound of lut_ptr[B] over the batches.  Outputs per batch as described
 * above (out / lut_batch / lut_node rows in ascending node order, n_lut[0] = L).  A single batch is a launch with
 * n_batches = 1. */
typedef struct qot_lp_batch {
  const float* x;              /* [N,5]                                       */
  const int64_t* edge_index;   /* [2,E]: source row, destination row          */
  const int64_t* ptr;          /* [B+1] node offsets                          */
  const int64_t* edge_ptr;     /* [B+1] edge offsets                          */
  const int64_t* lut_ptr;      /* [B+1] readout-row offsets                   */
  int64_t N, E, B;
  float* out;                  /* [>= L,3]                                    */
  int64_t* lut_batch;          /* [>= L]                                      */
  int32_t* lut_node;           /* [>= L]                                      */
  int32_t* n_lut;              /* [1]                                         */
  int32_t* status;             /* [1]                                         */
  float* z;                    /* [>= L,20] scratch                           */
  int64_t tile0;               /* first tile of this batch inside the launch  */
  int64_t reserved;            /* pads the descriptor to 128 bytes (it is copied as eight 16-byte pieces); 0 */
} qot_lp_batch_t;
/* flags: QOT_LP_SYMMETRIC_BY_SOURCE -- the caller has VERIFIED, for every graph of every batch of the launch,
 * the layout torch_geometric.utils.from_networkx gives an undirected nx.Graph (lightpath_training/dataset.py:86,
 * SURVEY.md A.6): edges grouped by source node ascending, every edge present in both directions, no duplicate
 * (source, destination) pair (PackedGraphStore.verify_layout does the check once per store).  The sources of a
 * node's in-edges are then the destinations of its own out-run, which the kernel locates by counting over the
 * destination row alone: the source row of edge_index is never read.  Same rows, bit-identical values. */
#define QOT_LP_SYMMETRIC_BY_SOURCE 1
/* QOT_LP_SPLIT_HEAD: run the readout head as a second launch (lp_stream_head_kernel, mma.sync) over z rows
 * written to the batches' workspaces, instead of inside the persistent kernel on tcgen05 / TMEM (the default). */
#define QOT_LP_SPLIT_HEAD 2
int64_t qot_lightpath_stream_tiles(int64_t B);
int qot_lightpath_infer_stream(const qot_lp_batch_t* batches, int32_t n_batches, int64_t total_tiles,
                               int64_t uniform_tiles, int64_t max_rows, const float* prepared,
                               int32_t is_lut_index, int32_t flags, void* stream);

/* Every-node mode (csrc/lightpath_every_node.cu, lp_every_node_kernel): every node of every graph evaluated as the
 * LUT, one pass over each graph.  For a batch with N nodes, row i of out [N,3] is what the reference
 * LightpathGNN.forward under eval() returns for node i's graph, given a copy of that graph in which node i's flag
 * column x[:, is_lut_index] is 1.0 and every other node's flag column is 0.0.  Whatever the stored flag column holds
 * has no effect.  Rows are in node order; the graph of row i is batch[i].
 * Same descriptor array as qot_lightpath_infer_stream, with tile0 counted in qot_lightpath_every_node_tiles(B) units.
 * Reads x, edge_index, ptr, edge_ptr, N, E, B, out (>= N rows), status (ZERO on entry; bit 0: malformed graph
 * offsets, the graph's rows are not written) and tile0; ignores lut_ptr / lut_batch / lut_node / n_lut / z, which
 * may be NULL.  `prepared` as for qot_lightpath_infer_stream (qot_lightpath_prepare); flags: 0 or
 * QOT_LP_SYMMETRIC_BY_SOURCE (same bits either way on a verified layout).  No host synchronisation: capturable. */
int64_t qot_lightpath_every_node_tiles(int64_t B);
int qot_lightpath_infer_every_node(const qot_lp_batch_t* batches, int32_t n_batches, int64_t total_tiles,
                                   int64_t uniform_tiles, const float* prepared, int32_t is_lut_index,
                                   int32_t flags, void* stream);

/* The evaluation loop of lightpath_training/test.py:77-94 for batches arriving from the HOST: one call per batch
 * replaces `data.to(device)` -> `model(data)` -> `.cpu()`.  The batch travels in the COMPACT WIRE FORMAT of a
 * verified-layout batch (see QOT_LP_SYMMETRIC_BY_SOURCE; PackedGraphStore.host_wire_batch packs it), one contiguous
 * pinned arena of qot_lightpath_wire_bytes(N, E, B, L) bytes:
 *   int32 ptr[B+1] | int32 edge_ptr[B+1] | int32 lut_ptr[B+1] | pad to 16 | float x4[N,4] | pad to 16 |
 *   uint8 lut_local[L] | pad to 16 | uint8 dst[E]
 * (x4: the node features without the LUT flag column, which must hold exactly 0.0 / 1.0 and travels as lut_local, the
 * graph-local node index of every readout row in row order; dst: graph-local destination id of every edge, graphs of
 * <= 255 nodes; no source row).  On `stream`: ONE host->device copy of the arena; lp_wire_unpack_kernel rebuilds the
 * reference layout in the slot (x [N,5], int64 edge_index [2,E], int64 offsets) and fills the slot's descriptor; the
 * status word is cleared; lp_stream_kernel (the same kernel resident
 * batches take: bit-identical rows); ONE device->host copy of the result arena [status | out rows | lut_batch rows],
 * L = lut_ptr[B] (known on the host).  No synchronisation: the caller waits on its own event.
 * h2d_bytes / d2h_bytes (optional, host): bytes this call copied in each direction. */
typedef struct {
  void* arena;            /* qot_lightpath_wire_bytes(cap_nodes, cap_edges, cap_graphs, cap_nodes) bytes, 16-byte aligned */
  float* x;               /* [cap_nodes, 5] -- rebuilt on the device                                           */
  int64_t* edge_index;    /* [2, cap_edges] -- rebuilt on the device                                           */
  int64_t* ptrs;          /* [3 * (cap_graphs + 1)]                                                            */
  qot_lp_batch_t* desc;   /* ONE descriptor in device memory, 16-byte aligned; the caller sets lut_node, n_lut and z
                             once (the slot's own buffers), the call fills the rest                             */
  void* result;           /* qot_lightpath_wire_result_bytes(cap_nodes) bytes, 16-byte aligned:
                             [status int32, 16 bytes | out [L,3] fp32 | pad to 16 | lut_batch [L] int64]         */
  int32_t* lut_node;      /* [cap_rows]                                                                        */
  int32_t* n_lut;         /* [1]                                                                               */
  int64_t cap_nodes, cap_edges, cap_graphs;
} qot_lp_wire_slot_t;
size_t qot_lightpath_wire_bytes(int64_t N, int64_t E, int64_t B, int64_t L);
size_t qot_lightpath_wire_result_bytes(int64_t L);
/* result_host: pinned, qot_lightpath_wire_result_bytes(L) bytes, same layout as slot->result (ONE device->host copy). */
int qot_lightpath_infer_wire_host(const void* arena_host, int64_t N, int64_t E, int64_t B, int64_t L,
                                  const float* prepared, int32_t is_lut_index, const qot_lp_wire_slot_t* slot,
                                  void* result_host, int64_t* h2d_bytes, int64_t* d2h_bytes, void* stream);

/* General GATConv forward over a destination-sorted CSR built with flags=3
 * (self loops replaced): h [N,128] = concat_h sum_j alpha_ij W_h x_j + bias.
 * Optional saves for the backward: z [N,4,5] = sum_j alpha_ij x_j per head, and the
 * softmax statistics smax [N,4], sden [N,4] (denominator incl. the 1e-16). */
int qot_gat_fwd(const float* x, const int32_t* rowptr, const int32_t* src, int64_t N,
                const float* lin_w, const float* att_src, const float* att_dst,
                const float* conv_bias, float* h, float* z, float* smax, float* sden,
                void* stream);

/* Backward of qot_gat_fwd w.r.t. its parameters (x carries no gradient: it is the
 * dataset input, lightpath_training/models.py:27): d_lin_w [128,5], d_att_src
 * [4,32], d_att_dst [4,32], d_bias [128]. */
size_t qot_gat_bwd_workspace_bytes(int64_t N);
int qot_gat_bwd(const float* x, const int32_t* rowptr, const int32_t* src, int64_t N,
                const float* lin_w, const float* att_src, const float* att_dst,
                const float* z, const float* smax, const float* sden, const float* dh,
                float* d_lin_w, float* d_att_src, float* d_att_dst, float* d_bias,
                void* ws, size_t ws_bytes, void* stream);

/* BatchNorm1d training statistics over the node dimension: mean [C], var [C]
 * (biased); per-chunk (mean, M2) combined in a fixed order.  When running_mean /
 * running_var are given they are updated in place with `momentum` (unbiased
 * variance), as torch.nn.BatchNorm1d does in train(). */
size_t qot_bn_stats_workspace_bytes(int64_t N, int64_t C);
int qot_bn_stats(const float* h, int64_t N, int64_t C, float* mean, float* var,
                 float* running_mean, float* running_var, float momentum,
                 void* ws, size_t ws_bytes, void* stream);

/* BatchNorm as a stand-alone layer over all rows (PyG BatchNorm, lightpath_training/models.py:31):
 * y = (x - mean) / sqrt(var + eps) * w + b with the given statistics (qot_bn_stats in train(),
 * running stats in eval()), and its dense backward: batch_stats=1 ->
 * dx = w*invstd*(dy - mean(dy) - xhat*mean(dy*xhat)); batch_stats=0 -> dx = w*invstd*dy;
 * d_w = sum(dy*xhat), d_b = sum(dy) (fixed-order two-stage sums).  C % 4 == 0. */
int qot_bn_apply(const float* x, int64_t N, int64_t C, const float* mean, const float* var,
                 float eps, const float* w, const float* b, float* y, void* stream);
size_t qot_bn_bwd_dense_workspace_bytes(int64_t N, int64_t C);
int qot_bn_bwd_dense(const float* x, const float* mean, const float* var, float eps, const float* w,
                     const float* dy, int64_t N, int64_t C, int batch_stats, float* dx, float* d_w,
                     float* d_b, void* ws, size_t ws_bytes, void* stream);

/* Ordered LUT compaction: lut_node [L] int32 ascending, lut_batch [L] int64
 * (optional), n_lut[0] = L  (lightpath_training/models.py:35-40). */
size_t qot_lut_select_workspace_bytes(int64_t N);
int qot_lut_select(const float* x, int64_t N, int64_t F, int32_t is_lut_index,
                   const int64_t* batch, int32_t* lut_node, int64_t* lut_batch,
                   int32_t* n_lut, void* ws, size_t ws_bytes, void* stream);

/* LUT rows: y = relu(bn(h[lut_node])) with the given statistics; hid = W1 y + b1;
 * out = W2 (leaky_relu(hid) * hmask) + b2.  hmask (optional [L,32]) is the dropout
 * keep-mask already divided by (1-p).  Saves y [L,128], hid [L,32] when non-NULL. */
int qot_lut_head_fwd(const float* h, const int32_t* lut_node, int64_t L,
                     const float* bn_mean, const float* bn_var, float bn_eps,
                     const float* bn_w, const float* bn_b, const float* W1, const float* b1,
                     const float* W2, const float* b2, const float* hmask, float* y,
                     float* hid, float* out, void* stream);

/* Backward of the head: dy [L,128] (gradient w.r.t. the BN output, ReLU mask
 * applied), dW1 [32,128], db1 [32], dW2 [3,32], db2 [3]. */
size_t qot_lut_head_bwd_workspace_bytes(int64_t L);
int qot_lut_head_bwd(const float* dout, const float* y, const float* hid, const float* hmask,
                     int64_t L, const float* W1, const float* W2, float* dy, float* dW1,
                     float* db1, float* dW2, float* db2, void* ws, size_t ws_bytes,
                     void* stream);

/* BatchNorm backward with a row-sparse upstream gradient (only LUT rows carry dy).
 * batch_stats=1 (train): dh [N,C] = g*invstd*(dy_n - mean(dy) - xhat_n*mean(dy*xhat));
 * batch_stats=0 (running stats): dh = g*invstd*dy_n.  Also d_bn_w [C], d_bn_b [C]. */
size_t qot_bn_bwd_workspace_bytes(int64_t N, int64_t L, int64_t C);
int qot_bn_bwd_sparse(const float* h, const float* mean, const float* var, float eps,
                      const float* bn_w, const float* dy, const int32_t* lut_node,
                      int64_t L, int64_t N, int64_t C, int batch_stats, float* dh,
                      float* d_bn_w, float* d_bn_b, void* ws, size_t ws_bytes, void* stream);

/* ---- graph construction on the device (SURVEY 8(f)4) -----------------------------------------
 * Replaces to_graph.py::create_lightpath_graph (to_graph.py:187-312: occupied-channel scan, one node
 * per conn_id in order of first appearance, node features from that first channel, is_lut = osnr ==
 * snr == ber == -1, interaction edges between lightpaths that share a link at 0 < |df| < threshold,
 * links used by a single lightpath skipped) fused with the tensorisation of
 * lightpath_training/dataset.py:53-123 (min-max scaling in fp64 then fp32, x columns in sorted-name
 * order [freq, is_lut, mod_order, num_spans, path_len], y = scaled [osnr, snr, ber]).
 * One thread block per sample; output is the packed graph store qot_collate consumes.
 *   data    [S, F, L, Q] float32, 0 = free channel          freqs [Q] float64 (the dataset's grid)
 *   target  [S, T] float64
 * Two launches, the sample tensor is read once: qot_lightpath_graph_count scans every sample, fills
 * counts [S,2] int32 = (nodes, directed edges), y [S,3] and a per-sample record in `scratch`
 * (qot_lightpath_graph_scratch_bytes(S) bytes, 16-byte aligned: node rows, conn ids, adjacency bits);
 * the caller scans the counts into node_ptr / edge_ptr [S+1] int64 and calls
 * qot_lightpath_graph_fill, which packs the records into node_feat [N_tot,5], conn_ids [N_tot] int64,
 * edge_src / edge_dst [E_tot] int32 (graph-local, both directions of every interaction, a self loop
 * once, sorted by (source, target) -- the reference's own edge ORDER follows CPython set iteration and
 * is not part of the contract).  status (int32[1], zeroed by the caller): bit 0 = a sample exceeds the
 * per-block capacities (QOT_TG_MAX_CHANNELS occupied channels, QOT_TG_MAX_NODES lightpaths, L <=
 * QOT_TG_MAX_LINKS); such a sample is reported with zero nodes; bit 1 = node_ptr / edge_ptr do not
 * match the records. */
#define QOT_TG_MAX_CHANNELS 6144
#define QOT_TG_MAX_NODES 256
#define QOT_TG_MAX_LINKS 1024
typedef struct {
  int32_t F, L, Q, T;              /* lp_feat, link, freq extents of `data`; columns of `target`          */
  int32_t i_conn, i_osnr, i_snr, i_ber;   /* rows of the lp_feat axis                                    */
  int32_t i_feat[4];               /* lp_feat rows of freq, mod_order, num_spans, path_len (x cols 0,2,3,4) */
  double feat_lo[4], feat_hi[4];   /* constants.py FEATURE_RANGES in the same order                       */
  int32_t i_tgt[3];                /* columns of `target` holding osnr, snr, ber                           */
  double tgt_lo[3], tgt_hi[3];     /* constants.py TARGET_RANGES                                           */
  double freq_threshold;           /* to_graph.py:188 (0.05)                                               */
} qot_lp_graph_cfg_t;
size_t qot_lightpath_graph_scratch_bytes(int64_t S);
int qot_lightpath_graph_count(const float* data, const double* freqs, const double* target, int64_t S,
                              const qot_lp_graph_cfg_t* cfg, int32_t* counts, float* y, void* scratch,
                              size_t scratch_bytes, int32_t* status, void* stream);
int qot_lightpath_graph_fill(const void* scratch, int64_t S, const int64_t* node_ptr,
                             const int64_t* edge_ptr, float* node_feat, int64_t* conn_ids,
                             int32_t* edge_src, int32_t* edge_dst, int32_t* status, void* stream);

/* Candidate QoT (csrc/lightpath_candidates.cu): candidate lightpaths evaluated against a resident NETWORK STATE -- raw
 * samples data [S, F, L, Q] float32 (0 = free channel), the grid freqs [Q] float64 and the qot_lp_graph_cfg_t they
 * were turned into graphs with (qot_lightpath_graph_count / _fill, then qot_collate of all S samples in order) --
 * without rebuilding the state's graphs.
 *
 * qot_lightpath_channel_map (lp_channel_map_kernel, once per state): chan_node [S, L, Q] int32 = the state-batch node
 * index of the lightpath on each channel, -1 on a free channel.  A channel is occupied when any of its F features is
 * non-zero; its lightpath is the conn_id row truncated toward zero (both as qot_lightpath_graph_count reads them),
 * looked up in conn_ids [N] int64 over the sample's nodes [node_ptr[s], node_ptr[s+1]) (node_ptr [S+1] int64).
 * status (optional, int32[1], zeroed by the caller): bit 0 = an occupied channel whose conn_id the sample's node list
 * lacks, or malformed node offsets; such a channel holds INT_MIN (occupied, no neighbour). */
int qot_lightpath_channel_map(const float* data, int64_t S, const qot_lp_graph_cfg_t* cfg, const int64_t* node_ptr,
                              const int64_t* conn_ids, int64_t N, int32_t* chan_node, int32_t* status, void* stream);

/* The five network-state queries below take the state and their inputs as host structs (read during the call, not
 * retained); the pointers in them are device pointers.
 *
 * A resident network state: the S samples' graphs collated in sample order (to_graph.lightpath_network_state).  x
 * [N,5], node_ptr [S+1], rowptr [N+1] int64 (node v's out-edges are [rowptr[v], rowptr[v+1]) of edge_index [2,E]
 * int64, which must be the layout qot_lightpath_graph_fill produces: sorted by source, every edge in both directions,
 * so a node's in-neighbours are the destinations of its out-run), chan_node from qot_lightpath_channel_map.  With S ==
 * 0 the arrays may be NULL; edge_index may be NULL when E == 0. */
typedef struct {
  qot_lp_graph_cfg_t cfg;      /* the configuration the graphs were built with, by value                    */
  int64_t S, N, E;
  const double* freqs;         /* [Q]                                                                       */
  const float* x;              /* [N,5]                                                                     */
  const int64_t* node_ptr;     /* [S+1]                                                                     */
  const int64_t* rowptr;       /* [N+1]                                                                     */
  const int64_t* edge_index;   /* [2,E]                                                                     */
  const int32_t* chan_node;    /* [S,L,Q]                                                                   */
  const int64_t* conn_ids;     /* [N]; read by qot_lightpath_provision only, may be NULL elsewhere          */
} qot_lp_state_t;              /* 264 bytes */

/* Candidates, reconfigurations and change-set changes: K of them, change k naming sample[k], the path
 * links[link_ptr[k] .. link_ptr[k+1]) (n_links entries of links in all), the slots [q0[k], q0[k] + width[k]) and the
 * raw channel vector feat[k]; node[k] is the lightpath a change moves. */
typedef struct {
  int64_t K, n_links;
  const int64_t* node;         /* [K]; ignored by qot_lightpath_candidates                                  */
  const int64_t* sample;       /* [K]                                                                       */
  const int64_t* link_ptr;     /* [K+1]                                                                     */
  const int32_t* links;        /* [n_links]                                                                 */
  const int32_t* q0;           /* [K]                                                                       */
  const int32_t* width;        /* [K]                                                                       */
  const float* feat;           /* [K,4]                                                                     */
} qot_lp_changes_t;            /* 72 bytes */

/* Placement and provisioning demands: D of them, demand d naming sample[d] and the options [opt_ptr[d],
 * opt_ptr[d+1]); option p (P of them) is the route links[link_ptr[p] .. link_ptr[p+1]) (n_links entries in all), a
 * slot width, channel features and a bound on its own metric. */
typedef struct {
  int64_t D, P, n_links;
  const int64_t* sample;       /* [D]                                                                       */
  const int64_t* opt_ptr;      /* [D+1]                                                                     */
  const int64_t* link_ptr;     /* [P+1]                                                                     */
  const int32_t* links;        /* [n_links]                                                                 */
  const int32_t* width;        /* [P]                                                                       */
  const float* feat;           /* [P,3]                                                                     */
  const float* own_bound;      /* [P]                                                                       */
} qot_lp_demands_t;            /* 80 bytes */

/* qot_lightpath_candidates (lp_candidate_kernel): K candidates, one warp each, one launch.  Candidate k names sample
 * sample[k], a path links[link_ptr[k] .. link_ptr[k+1]) (int32 link indices; duplicates change nothing), the slot
 * range [q0[k], q0[k] + width[k]) used on every link of the path and its raw channel vector feat [K,4] = (freq,
 * mod_order, num_spans, path_len), the values to_graph would read from its channels.  sample' = data[sample[k]] with
 * the candidate written into every channel of its path and slot range (new conn_id, features feat[k], osnr = snr =
 * ber = -1).  In sample''s lightpath graph, with the flag column x[:, is_lut_index] one-hot:
 *   out [K,3]          row k: the reference LightpathGNN.forward under eval() with the flag at the candidate's node;
 *   impact rows        one per existing lightpath j adjacent to the candidate (sharing a link at 0 < |freqs[qc] -
 *                      freqs[qj]| < cfg.freq_threshold in fp64): the same forward with the flag at j, in ascending
 *                      order of j's state-batch node index.  impact_node [K,max_impact] int64 = j, impact_out
 *                      [K,max_impact,3]; slots past the rows written hold -1 / NaN.  n_impact [K] int32 = the number
 *                      of neighbours (may exceed max_impact).
 * Candidates are independent of each other.  The candidate's x row is feat scaled as qot_lightpath_graph_count scales
 * node features (min-max in fp64 of the float32 value with cfg.feat_lo / feat_hi, then fp32).  `prepared` as for
 * qot_lightpath_infer_stream.  status [K] int32 (written for every candidate), bits QOT_CAND_*: with BAD_SAMPLE,
 * BAD_PATH, OCCUPIED or BAD_STATE before the scan ends the out row is NaN and n_impact is 0; with IMPACT_OVERFLOW the
 * out row and the first max_impact impact rows are written.  No host synchronisation: capturable; a malformed
 * candidate never faults and never stops the launch. */
#define QOT_CAND_BAD_SAMPLE 1        /* sample[k] outside [0, S)                                                  */
#define QOT_CAND_BAD_PATH 2          /* empty path, a link outside [0, L), width < 1 or slot range outside [0, Q) */
#define QOT_CAND_OCCUPIED 4          /* a channel of the candidate is occupied on some link of its path           */
#define QOT_CAND_IMPACT_OVERFLOW 8   /* more neighbours than max_impact                                           */
#define QOT_CAND_BAD_STATE 16        /* the state arrays are inconsistent (offsets, chan_node, rowptr); the
                                        affected rows are NaN                                                     */
int qot_lightpath_candidates(const qot_lp_state_t* state, const qot_lp_changes_t* cands, const float* prepared,
                             int32_t is_lut_index, int32_t max_impact, float* out, int32_t* status, int32_t* n_impact,
                             int64_t* impact_node, float* impact_out, void* stream);

/* qot_lightpath_reconfigure (lp_candidate_kernel, the same launch shape): K changes to the state, evaluated
 * independently, each against the state alone.  Change k takes the candidate arguments above plus node [K] int64:
 * the lightpath it moves, a node of the state batch in [node_ptr[s], node_ptr[s+1]) for s = sample[k], or -1 for a
 * plain insertion (then every output is bit-identical to qot_lightpath_candidates and every impact_kind is 2).  Let c
 * be the moved lightpath j's conn_id.  sample' = data[s] with every channel of conn_id c zeroed and then, unless the
 * change is a teardown, one vector written on every channel of the path and slot range: conn_id c, the feat[k] values,
 * and j's other rows (src/dst, metrics) from j's first channel.  AN EMPTY PATH WITH node[k] >= 0 IS A TEARDOWN, not
 * BAD_PATH: q0, width and feat are not read, the out row is NaN.  A channel of the new placement is occupied when its
 * chan_node is neither -1 nor j (j's own channels are free; INT_MIN is occupied).  In sample''s graph:
 *   out [K,3]          the forward with the flag at j's new node (NaN for a teardown);
 *   impact rows        every lightpath i != j that was adjacent to j in the state graph or is adjacent to j in
 *                      sample''s graph, ascending in node order of the state batch: impact_node = i, impact_out = the
 *                      forward with the flag at i, impact_kind [K,max_impact] int8 (optional, may be NULL) = bit 0: i
 *                      was j's neighbour, bit 1: i is j's neighbour after the change (1 lost j, 2 gained j, 3 kept j
 *                      with its new features); slots past the rows written hold -1 / 0 / NaN.  n_impact [K] = the
 *                      number of such rows (may exceed max_impact).
 * Every other row of sample' equals its row in the state.  Message order: j's row = its new neighbours ascending, then
 * its self loop; row i = i's state in-row ascending without j and without i's self loop, then j if bit 1 is set, then
 * i's self loop.  Status bits QOT_CAND_*, plus BAD_NODE; with BAD_NODE the out row is NaN and n_impact is 0. */
#define QOT_CAND_BAD_NODE 32         /* node[k] is neither -1 nor a node of sample[k]                             */
int qot_lightpath_reconfigure(const qot_lp_state_t* state, const qot_lp_changes_t* changes, const float* prepared,
                              int32_t is_lut_index, int32_t max_impact, float* out, int32_t* status, int32_t* n_impact,
                              int64_t* impact_node, int8_t* impact_kind, float* impact_out, void* stream);

/* qot_lightpath_change_sets (lp_change_set_kernel, the same launch shape, one warp per set): G sets of changes, each
 * evaluated jointly against the state.  The changes take the qot_lightpath_reconfigure arguments; set g is changes
 * [set_ptr[g], set_ptr[g+1]) (set_ptr [G+1] int64), all naming one sample s, at most QOT_SET_MAX_CHANGES of them.
 * sample' = data[s] with (1) every channel of every lightpath the set moves or tears down (node >= 0) zeroed, then
 * (2) each non-teardown change written on its path x slot range: a move as qot_lightpath_reconfigure writes it (j's
 * conn_id, feat, j's other rows from its first channel), an insertion with a new conn_id (one above the sample's
 * largest, +1 per insertion in set order; metrics -1).  The placements of a set must be disjoint.  A channel is occupied
 * only when its chan_node is a lightpath the set does not move (so swaps are legal; INT_MIN is occupied).  In sample''s
 * graph, flag one-hot:
 *   out [K,3]            the changed lightpath's row at its new placement; NaN for a teardown;
 *   impact rows          per set, every lightpath i of the state that the set does not move and that is adjacent to a
 *                        changed lightpath before or after the set, ascending in node order of the state batch:
 *                        impact_node [G,M], impact_out [G,M,3], impact_kind [G,M] int8 (may be NULL) = bit 0: an
 *                        in-neighbour of i is moved or torn down, bit 1: a changed lightpath is i's neighbour after the
 *                        set; past the rows -1 / 0 / NaN.  n_impact [G] = the number of such rows (may exceed M).
 * Every other row of sample' equals its row in the state.  Message order: the row of change c = its new neighbours in
 * the state ascending, then the other changes adjacent to it in set order, then its self loop; impact row i = i's state
 * in-row ascending without the removed lightpaths and without i's self loop, then the changes adjacent to i in set
 * order, then i's self loop.  A set of one change is bit-identical to qot_lightpath_reconfigure.
 * status [K] = the QOT_CAND_* bits of each change plus the QOT_SET_* bits below (IMPACT_OVERFLOW on every change of an
 * overflowing set, BAD_STATE found in an impact row on the set's first change); set_status [G] = the OR over the set.
 * Every bit but IMPACT_OVERFLOW is fatal for the whole set: all its out rows are NaN and n_impact is 0.  If set_ptr is
 * not non-decreasing from 0 to K, no set is evaluated: every status and set_status is BAD_SET. */
#define QOT_SET_MAX_CHANGES 64
#define QOT_SET_BAD_SET 64           /* the set's changes name different samples (on the changes that differ from the
                                        first), the set has more than 64 changes, or set_ptr is malformed            */
#define QOT_SET_DUPLICATE 128        /* a lightpath is moved or torn down by two changes of the set (on both)       */
#define QOT_SET_CONFLICT 256         /* this change's placement shares a channel with another change's placement    */
int qot_lightpath_change_sets(const qot_lp_state_t* state, const qot_lp_changes_t* changes, int64_t G,
                              const int64_t* set_ptr, const float* prepared, int32_t is_lut_index, int32_t max_impact,
                              float* out, int32_t* status, int32_t* set_status, int32_t* n_impact,
                              int64_t* impact_node, int8_t* impact_kind, float* impact_out, void* stream);

/* qot_lightpath_placements (lp_placement_kernel, the same launch shape, one warp per demand): D demands, each a sample
 * sample[d] and options [opt_ptr[d], opt_ptr[d+1]) (opt_ptr [D+1] int64, 1..QOT_PLACE_MAX_OPTIONS options).  Option p
 * (P of them) is a route links[link_ptr[p] .. link_ptr[p+1]) (link_ptr [P+1] int64), a slot width width[p], channel
 * features feat [P,3] = (mod_order, num_spans, path_len) and a bound own_bound [P] on its own metric.  A placement is
 * an option with a start slot q0 in [0, Q - width] whose channels [q0, q0 + width) are free (chan_node -1) on every
 * link of the route; its rows are, by definition, the qot_lightpath_candidates rows of the candidate (sample, route,
 * q0, width, feat = (float32(freqs[q0]), mod_order, num_spans, path_len)).  A row's margin (fp32, round to nearest)
 * is v - b if maximize, else b - v, with v its output column `metric` (0..2) and b own_bound[p] for the own row or
 * bound[node] (bound [N] float32, may be NULL: impact rows unconstrained) for each impact row, every impact row
 * counted whatever max_impact is.  A placement's margin is the minimum over its rows (NaN if one is NaN); it is
 * feasible iff the margin is >= 0.  Among the feasible placements `policy` picks one, a tie going to the lower option
 * and then the lower q0:
 *   QOT_PLACE_FIRST_FIT    the first in (option, q0) order;
 *   QOT_PLACE_BEST_QOT     the best own value (highest if maximize, lowest otherwise);
 *   QOT_PLACE_MAX_MARGIN   the largest margin.
 * Outputs per demand: option / q0 [D] int32 (option relative to opt_ptr[d]; -1 / -1 if none is feasible), out [D,3]
 * the chosen own row (NaN if none), margin [D] (NaN if none), n_free / n_feasible [D] int32 over every placement of
 * the demand, status [D] int32, and the chosen placement's n_impact / impact_node [D,max_impact] / impact_out
 * [D,max_impact,3] exactly as qot_lightpath_candidates lays them out.  all_out [P,Q,3] / all_margin [P,Q] (both NULL,
 * or both given): every free placement's own row and margin, NaN at every other (option, q0) of a demand's options.
 * Status bits QOT_CAND_*: BAD_SAMPLE; BAD_PATH (an empty route, a link outside [0, L), a width outside [1, Q), zero
 * or more than QOT_PLACE_MAX_OPTIONS options, a malformed opt_ptr or link_ptr range); BAD_STATE (a route's channel
 * holds a node outside the sample, a bad in-row); IMPACT_OVERFLOW (the chosen placement has more than max_impact
 * impact rows).  Any bit but IMPACT_OVERFLOW: option = q0 = -1, NaN rows, zero counts.  Q <= QOT_PLACE_MAX_SLOTS.
 * No host synchronisation: capturable; a malformed demand never faults and never stops the launch. */
#define QOT_PLACE_MAX_OPTIONS 32
#define QOT_PLACE_MAX_SLOTS 1024
#define QOT_PLACE_FIRST_FIT 0
#define QOT_PLACE_BEST_QOT 1
#define QOT_PLACE_MAX_MARGIN 2
int qot_lightpath_placements(const qot_lp_state_t* state, const qot_lp_demands_t* demands, const float* bound,
                             int32_t metric, int32_t maximize, int32_t policy, const float* prepared,
                             int32_t is_lut_index, int32_t max_impact, int32_t* option, int32_t* q0, float* out,
                             float* margin, int32_t* n_free, int32_t* n_feasible, int32_t* status, int32_t* n_impact,
                             int64_t* impact_node, float* impact_out, float* all_out, float* all_margin, void* stream);

/* qot_lightpath_provision (lp_provision_kernel, one block per sample, persistent over samples): sequential
 * provisioning.  The demands and arguments of qot_lightpath_placements, plus order [D] / sample_ptr [S+1] int64, the
 * demands grouped by sample: sample s's demands are order[sample_ptr[s] .. sample_ptr[s+1]), ascending, and the
 * ranges hold every demand whose sample lies in [0, S).  Samples are independent; the demands of one sample are
 * provisioned in that order, demand d placed exactly as qot_lightpath_placements places it against state_d, the state
 * built from the samples with every earlier accepted demand of d's sample written in.  An accepted demand is written
 * as qot_lightpath_candidates writes a candidate: its chosen option's route x [q0, q0 + width), conn_id one above the
 * sample's largest (top + 1, top + 2, ... for successive acceptances; conn_ids [N] is the state's), freq =
 * float32(freqs[q0]), the option's (mod_order, num_spans, path_len), osnr = snr = ber = -1.  With a bound, an accepted
 * demand's impact rows are bound from then on by its option's own_bound.  A demand is accepted when it has a feasible
 * placement and no status bit but IMPACT_OVERFLOW; otherwise it commits nothing and the sample's later demands go on.
 * Outputs per demand as qot_lightpath_placements (no all_out / all_margin), bit-identical to its result against
 * state_d, except: impact_conn [D, max_impact] int64 names the impact rows by conn_id (-1 past the rows), and conn_id
 * [D] int64 is the id the demand was accepted under (-1: not accepted).  Status bits QOT_CAND_* as there, plus:
 *   QOT_PROV_FULL           accepting would take the sample past QOT_TG_MAX_NODES lightpaths or QOT_TG_MAX_CHANNELS
 *                           occupied channels (the graph builder refuses such a sample): not accepted, the placement
 *                           is still reported;
 *   QOT_PROV_BAD_GROUPING   order / sample_ptr are not such a grouping: no demand is provisioned, every demand gets
 *                           this status alone, -1 / NaN rows and zero counts.
 * A demand whose sample lies outside [0, S) gets BAD_SAMPLE.  Work arrays: chan_work [S, L, Q] int32 (the entry point
 * copies chan_node into it, the kernel writes the accepted channels) and bound_work [S, QOT_TG_MAX_NODES] float32
 * (required with a bound, else unused).  The state is not modified.  One copy and one launch, nothing read back:
 * capturable; a malformed demand or grouping never faults and never stops the launch. */
#define QOT_PROV_FULL 512
#define QOT_PROV_BAD_GROUPING 1024
int qot_lightpath_provision(const qot_lp_state_t* state, const qot_lp_demands_t* demands, const int64_t* order,
                            const int64_t* sample_ptr, const float* bound, int32_t metric, int32_t maximize,
                            int32_t policy, const float* prepared, int32_t is_lut_index, int32_t max_impact,
                            int32_t* chan_work, float* bound_work, int32_t* option, int32_t* q0, float* out,
                            float* margin, int32_t* n_free, int32_t* n_feasible, int32_t* status, int32_t* n_impact,
                            int64_t* conn_id, int64_t* impact_conn, float* impact_out, void* stream);

/* The topological representation: to_graph.py::create_topological_graph (:62-184: one edge per
 * lightpath between its source and destination network node, lightpaths added in ascending conn_id,
 * nx.Graph keeps one edge per node pair -- position from the first, attributes from the last) fused
 * with topological_training/dataset.py:46-123 (relabelling copy, from_networkx edge order, min-max
 * scaled edge_attr in sorted-name order [freq, mod_order, num_spans, path_len], y).  Every sample has
 * num_nodes nodes (75, to_graph.py:134; node_ptr = num_nodes * s, no node features).  Same two-launch
 * protocol (scan into `scratch` + counts [S] int32 = directed edges per sample and y; then pack):
 * edge_src / edge_dst [E_tot] int32 in
 * the REFERENCE'S edge order, edge_feat [E_tot,4], y [S,3].  i_src / i_dst: lp_feat rows of src_id /
 * dst_id (1-based node ids).  status bit 0: capacity exceeded or an endpoint outside 1..num_nodes. */
size_t qot_topological_graph_scratch_bytes(int64_t S);
int qot_topological_graph_count(const float* data, const double* target, int64_t S,
                                const qot_lp_graph_cfg_t* cfg, int32_t num_nodes, int32_t i_src,
                                int32_t i_dst, int32_t* counts, float* y, void* scratch,
                                size_t scratch_bytes, int32_t* status, void* stream);
int qot_topological_graph_fill(const void* scratch, int64_t S, const int64_t* edge_ptr,
                               int32_t* edge_src, int32_t* edge_dst, float* edge_feat,
                               int32_t* status, void* stream);

/* ---- TopologicalGNN, one block per graph (csrc/topo_fused.cu) -----------------------------------
 * The whole forward of topological_training/models.py:43-64 in one launch and the whole backward
 * (forward recomputed, every parameter gradient) in another, for the reference shape (hidden 16,
 * edge_dim 4, edge MLP 4 -> 8 -> 256, 3 outputs, embedding branch, dropout inactive) and graphs small
 * enough for one block's shared memory.  `flat` [qot_topo_fused_params()] fp32: Wq bq Wk bk Wv bv Ws bs
 * We | nn.0.weight nn.0.bias nn.2.weight nn.2.bias | conv2.lin.weight conv2.bias | mlp.0.weight
 * mlp.0.bias mlp.3.weight mlp.3.bias, each row-major as in the state_dict; qot_topo_fused_prepare
 * turns it into `prepared` [qot_topo_fused_prepared_floats()] (transposed copies, factorised NNConv
 * layout) once per weight update -- the kernels read that 22 KB buffer through L1; emb [num_nodes,16].
 * nmax / emax: largest node / edge count of a graph in the batch (host-known from the collate).
 * Forward: out [B,3]; `saved` (optional, qot_topo_fused_saved_floats(N, E, B) floats): the forward
 * state the backward would otherwise recompute (q k v h1 h2 T per node, edge-MLP hidden + softmax
 * weights per edge).  Backward: dout [B,3] (+ the same `saved`, or NULL to recompute) -> gflat (same
 * layout as flat), gemb [num_nodes,16]; ws: qot_topo_fused_bwd_workspace_bytes(num_nodes).
 * N = total nodes of the batch.  Deterministic (fixed summation orders).
 * Dropout (models.py:55,59 on the node features; :36-41 in the head) takes its masks as an INPUT: drop_mask,
 * one byte per element -- [N,16] after conv1 | [N,16] after conv2 | [B,16] inside the head, 1 = keep -- drawn by
 * the caller (torch's generator, so CUDA-graph replays advance it and tests can replay the masks through the
 * oracle); kept elements are scaled by drop_scale = 1 / (1 - p) (drop_scale_head in the head).  NULL = no
 * dropout; the backward takes the same mask.
 * status bit 0: a graph exceeds nmax / emax (skipped; its output is NaN), bit 1: a node id or edge endpoint out
 * of range (clamped). */
int qot_topo_fused_params(void);
int qot_topo_fused_prepared_floats(void);
int qot_topo_fused_prepare(const float* flat, float* prepared, void* stream);
size_t qot_topo_fused_saved_floats(int64_t N, int64_t E, int64_t B);
int qot_topo_fused_fwd(const float* prepared, const float* emb, const int64_t* node_ids,
                       const int64_t* edge_index, int64_t E, const float* edge_attr,
                       const int64_t* gptr, const int64_t* eptr, int64_t B, int64_t N, int32_t nmax,
                       int32_t emax, int32_t num_nodes, float* out, float* saved, int32_t* status,
                       const uint8_t* drop_mask, float drop_scale, float drop_scale_head, void* stream);
size_t qot_topo_fused_bwd_workspace_bytes(int32_t num_nodes);
int qot_topo_fused_bwd(const float* prepared, const float* emb, const int64_t* node_ids,
                       const int64_t* edge_index, int64_t E, const float* edge_attr,
                       const int64_t* gptr, const int64_t* eptr, int64_t B, int64_t N, int32_t nmax,
                       int32_t emax, int32_t num_nodes, const float* dout, const float* saved, float* gflat,
                       float* gemb, void* ws, size_t ws_bytes, int32_t* status,
                       const uint8_t* drop_mask, float drop_scale, float drop_scale_head, void* stream);

/* ------------------------------------------------------------------------ */
/* Data-parallel training tail: gradient exchange + optimizer update, ONE launch.     */
/* The reference trains single-process (topological_training/train.py:107-116:        */
/* loss.backward(); optimizer.step(), torch.optim.SGD at :66); the multi-GPU split    */
/* with a gradient all-reduce is what BASELINE.json's north_star adds.                */
/* ------------------------------------------------------------------------ */
/* Flat gradient `grad` [n] of this rank (FlatGradBuffer order) -> one-shot all-reduce over NVLink peer memory ->
 * averaged gradient written back to `grad` -> torch.optim.SGD's update (weight decay, momentum, dampening, nesterov,
 * maximize) on `momentum_buf` [n] and the parameter tensors named by `segs`.
 *   peers   DEVICE array of `world` pointers: peers[r] = rank r's exchange buffer as mapped in THIS process (CUDA IPC
 *           or torch symmetric memory), qot_ddp_exchange_bytes(n) bytes each, zero-initialised once; NULL when
 *           world == 1.  Every rank must call with the same n and launch once per step.
 *   hyper   DEVICE struct: a captured step follows an lr schedule by updating it between replays.
 *   state   DEVICE, two 64-bit words, zero-initialised once: [0] steps taken (the flag value of the exchange -- never
 *           reset it on one rank only), [1] != 0 once the momentum buffer holds a gradient (clear it to make the next
 *           step clone the gradient into the buffer, as torch does for a fresh optimizer).
 *   status  bit 0: a peer did not arrive within 4 s (no update was applied).
 * Sums in rank order on every rank: the replicas stay bit-identical.
 * `one_minus_dampening` is the momentum update's gradient factor, 1 - dampening computed in double and rounded to
 * float once, as torch.optim.SGD passes it to its foreach kernels; float(1) - float(dampening) differs from it by one
 * ulp for dampening 0.6, 0.8, 0.9, 0.99 or 1/3, and the trajectory would leave torch's in the low bits.  `dampening` itself is
 * not read by the kernel. */
typedef struct {
  float* param;          /* the parameter tensor (fp32, contiguous)           */
  int64_t offset;        /* its first element in the flat gradient            */
  int64_t numel;
} qot_param_seg_t;
typedef struct {
  float lr, momentum, dampening, weight_decay;
  int32_t nesterov, maximize;
  float one_minus_dampening;
  int32_t reserved;
} qot_sgd_hyper_t;
size_t qot_ddp_exchange_bytes(int64_t n);
int qot_ddp_sgd_step(float* grad, float* const* peers, int32_t world, int32_t rank, int64_t n,
                     const qot_param_seg_t* segs, int32_t nseg, float* momentum_buf,
                     const qot_sgd_hyper_t* hyper, unsigned long long* state, int32_t* status, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* QOT_B200_H_ */
