/*
 * bigcn_b200 -- C-ABI of the B200-native BiGCN hot path (libbigcn_b200.so).
 *
 * Every entry point takes plain DEVICE pointers, sizes and a CUDA stream
 * (passed as void*, i.e. cudaStream_t).  Nothing here depends on torch.
 * Buffers are borrowed: the caller allocates inputs, outputs and workspaces
 * (sizes come from the *_bytes queries) and keeps them alive until the stream
 * has drained.  No entry point synchronises the host or allocates device memory.
 * bigcn_features_forward / _backward fork short independent kernels onto internal
 * streams (created on first use, per device) and join them again before they return:
 * at return all work is ordered on the caller's stream.  One exception: in
 * BIGCN_GEMM_SPARSE training the forward leaves the column sort of x running on a
 * low-priority stream and bigcn_features_backward waits for it where it needs it; the
 * workspace must outlive that (bigcn_join_internal_streams(stream) makes `stream` wait
 * for everything in flight; bigcn_internal_stream() is that stream's handle for
 * allocators that track per-stream use).  Calls are not re-entrant per device.
 * Return value: 0 = ok, non-zero = error (bigcn_last_error()).
 * Data-dependent input violations (edge endpoint >= N, unsorted batch, root
 * outside its tree) never produce a silent wrong answer: they raise bits in the
 * caller's device-side `flags` word, which the host reads at its next sync.
 *
 * The reference (cwkd/BiGCN, /root/reference) has no FFI: its hot path is the
 * nn.Module code of model/Twitter/BiGCN_Twitter.py:19-131 calling
 * torch_geometric.nn.GCNConv and torch_scatter.scatter_mean.  Each function
 * below cites the reference lines (and the library routine behind them) that
 * it replaces; INTEGRATION.md shows the ctypes binding a maintainer adds.
 *
 * Conventions: fp32 row-major; hid_feats == out_feats == 64 (the reference's
 * only configuration, BiGCN_Twitter.py:140-144); int64 index inputs exactly as
 * PyG hands them over, narrowed to int32 on the device (N, E < 2^31).
 */
#ifndef BIGCN_B200_H
#define BIGCN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BIGCN_H 64 /* hid_feats == out_feats */

/* flags word bits (device int32, OR-ed by kernels) */
#define BIGCN_FLAG_EDGE_RANGE 1   /* an edge endpoint is < 0 or >= N            */
#define BIGCN_FLAG_BATCH_ORDER 2  /* batch[] not sorted ascending / out of [0,B) */
#define BIGCN_FLAG_ROOT_RANGE 4   /* rootindex[b] outside [0,N)                 */
#define BIGCN_FLAG_X_NOT_SPARSE 8 /* BIGCN_GEMM_SPARSE on a batch with more non-zeros than N*min(K,48):
                                     the conv1 weight gradient is NaN, use a dense gemm_mode          */

#define BIGCN_FLAG_EDGE_WEIGHT 32  /* edge-weighted batch: a weight is not finite, or a node's weighted degree is
                                      negative (its deg^-1/2 would be NaN) */
#define BIGCN_FLAG_X_CSR_RANGE 16  /* sparse input: a column index of x is outside [0,K) (entry ignored) */

/* degree convention of gcn_norm: PyG 2.x sums at the target (col); the
 * readme-pinned 1.3.2 summed at the source (row). */
#define BIGCN_DEG_BY_TARGET 0
#define BIGCN_DEG_BY_SOURCE 1

/* X*W arithmetic: exact fp32 FFMA scan, or tcgen05 kind::tf32 with 1 / 2 / 3 MMAs per K step.
 * TF32X3: both operands split hi + lo (x_hi w_hi + x_hi w_lo + x_lo w_hi): fp32-class on ANY input; the x split
 *         happens in shared memory between the TMA load and the MMA, x is still read from HBM once.
 * TF32X2: only the small operand (W forward, T backward) is split: exact to ~2^-22 when x is representable in
 *         TF32 (bag-of-words counts are), one MMA less per K step. */
#define BIGCN_GEMM_FP32 0
#define BIGCN_GEMM_TF32 1
#define BIGCN_GEMM_TF32X3 2
#define BIGCN_GEMM_TF32X2 5
/* exact fp32 scan for X*W (forward), tcgen05 hi/lo-split GEMM for the weight gradient.  The weight gradient is the
 * TF32X2 product (T split, x as it is): like TF32X2 it is exact to ~2^-22 only when x is representable in TF32
 * (bag-of-words counts are); on dense features it is 1e-4-class, so use TF32X3 or FP32 there. */
#define BIGCN_GEMM_MIXED 3
/* exact fp32 scan forward that also captures the non-zeros of x; the weight gradient is a sweep
 * over the column-sorted non-zeros (no second pass over x).  For bag-of-words inputs. */
#define BIGCN_GEMM_SPARSE 4
/* x is a dense BF16 matrix: every `const float* x` of a call made in this mode (bigcn_batch_t.x, bigcn_xw,
 * bigcn_xw_wgrad, bigcn_gcnconv_forward / _backward) points at bf16 rows with a pitch of K elements; K must be a
 * multiple of 8 and x 16 B aligned (TMA).  X*W and dW1 run on tcgen05 kind::f16 with the small operand (W forward,
 * T backward) split into three bf16 terms (24 significant bits): fp32-class relative to the fp32 widening of x.
 * Parameters, activations and gradients stay fp32.  Not for CSR input or the edge-weighted GCNConv (error). */
#define BIGCN_GEMM_BF16 6

/* direction bits */
#define BIGCN_DIR_TD 1
#define BIGCN_DIR_BU 2

typedef void* bigcn_stream_t; /* cudaStream_t */

typedef struct bigcn_dims {
  int64_t N;    /* nodes in the batch                    */
  int64_t B;    /* trees in the batch (rootindex.numel())*/
  int64_t K;    /* in_feats                              */
  int64_t C;    /* classes of the head (4 / 2)           */
  int64_t E_td; /* columns of data.edge_index            */
  int64_t E_bu; /* columns of data.BU_edge_index         */
} bigcn_dims_t;

/* The five attributes forward(data) reads (BiGCN_Twitter.py:27,45-47,78). */
typedef struct bigcn_batch {
  const float* x;               /* [N,K]    data.x (bf16 rows in BIGCN_GEMM_BF16) */
  const int64_t* edge_index;    /* [2,E_td] data.edge_index  [parent;child] */
  const int64_t* bu_edge_index; /* [2,E_bu] data.BU_edge_index [child;parent] */
  const int64_t* batch;         /* [N]      data.batch (sorted)          */
  const int64_t* rootindex;     /* [B]      data.rootindex (global ids)  */
  int64_t node_id_base;         /* global id of local node 0: dropout masks are keyed on
                                   global ids so they do not depend on the world size */
  /* Sparse input (BIGCN_GEMM_SPARSE only, x == NULL): data.x as CSR, e.g. from a loader that
   * keeps the `index:count` pairs of Process/getTwittergraph.py:16-24 or from
   * bigcn_host_dense_to_csr.  Columns of a row must be distinct. */
  const int32_t* x_ptr;         /* [N+1]                                   */
  const int32_t* x_col;         /* [x_ptr[N]]                              */
  const float* x_val;           /* [x_ptr[N]]                              */
  /* NULL, or the buffer bigcn_batch_prepare filled for THIS batch (same dims, same pointers above): features_forward /
   * bigcn_train_tail / features_backward then skip graph prep, the root columns and -- BIGCN_GEMM_SPARSE -- the pass
   * over x (the product becomes a sweep over the prepared CSR, bit-identical to the fused scan). */
  void* prepared;
  /* NULL, or the weight of every edge of the direction ([E_td] / [E_bu] fp32, aligned with edge_index /
   * bu_edge_index): both convs of that direction then run GCNConv(x, edge_index, edge_weight) -- gcn_norm with weights
   * (a self-loop edge in the list hands its weight to the node's loop, the last one wins; fill 1 otherwise; degree =
   * the weighted sum).  NULL = the unweighted path, unchanged.  Needs a workspace of
   * bigcn_features_edge_workspace_bytes; a `prepared` buffer must then come from bigcn_batch_prepare on this batch with
   * these weight pointers and values (it carries the weighted normalisation, which opts.edge_grad then also reads). */
  const float* td_edge_weight;
  const float* bu_edge_weight;
} bigcn_batch_t;

/* Parameters in PyG-2.x state_dict layout (SURVEY.md 8b):
 *   <dir>.conv1.lin.weight [64,K], <dir>.conv1.bias [64],
 *   <dir>.conv2.lin.weight [64,64+K], <dir>.conv2.bias [64], fc.weight [C,256], fc.bias [C].
 * The same struct with non-const meaning is used for gradients. */
typedef struct bigcn_params {
  float* td_w1; float* td_b1; float* td_w2; float* td_b2;
  float* bu_w1; float* bu_b1; float* bu_w2; float* bu_b2;
  float* fc_w;  float* fc_b;
} bigcn_params_t;

/* Normalised structure of one direction, emitted instead of PyG's COO' list. */
typedef struct bigcn_graph {
  int32_t* in_ptr;  /* [N+1] CSR by target                                  */
  int32_t* in_idx;  /* [E]   sources of in-edges, edge-list (COO') order    */
  int32_t* out_ptr; /* [N+1] CSR by source (A-hat^T, used by backward)      */
  int32_t* out_idx; /* [E]   targets of out-edges, edge-list order          */
  int32_t* deg;     /* [N]   degree incl. the unit self-loop                */
  float* dis;       /* [N]   deg^-1/2 = 1.0f / sqrtf(deg), IEEE             */
  float* rowsum;    /* [N]   sum_j A-hat[i,j] in COO' order, or NULL        */
  int32_t* in_long; /* hub-row work list of the by-target CSR: bigcn_long_ws_ints(E) ints, or NULL */
  int32_t* out_long;/* same for the by-source CSR                                              */
} bigcn_graph_t;

typedef struct bigcn_opts {
  int32_t training;   /* module.training: dropout on/off (BiGCN_Twitter.py:54)      */
  float p_drop;       /* F.dropout default 0.5                                      */
  uint64_t seed;      /* Philox key                                                 */
  int32_t deg_by;     /* BIGCN_DEG_BY_*                                             */
  int32_t gemm_mode;  /* BIGCN_GEMM_*                                               */
  int32_t dir_mask;   /* BIGCN_DIR_TD | BIGCN_DIR_BU                                */
  int32_t bwd_phase;  /* features_backward: 0 all, 1 all but dW1, 2 dW1 only        */
  int32_t skip_wgrad_prep; /* BIGCN_GEMM_SPARSE forward: 1 = inference, do not sort the
                              non-zeros of x by column (features_backward would then
                              return NaN for the conv1 weight gradient)              */
  int32_t fused_tail; /* training step through bigcn_train_tail: features_forward leaves the second
                         readout pass, features_backward the gscale pass, to that one launch   */
  const uint64_t* seed_dev; /* NULL, or a device counter: the Philox key is seed + *seed_dev, read when the
                               kernels run.  bigcn_adam_step / bigcn_dp_reduce_adam advance step_count[2] once
                               per step, so a captured CUDA graph of the step draws fresh masks at every replay */
  int32_t dense_roots; /* training only: 1 = the root rows of x are dense (PHEME's sentence embeddings): the root half of
                          conv2.lin (BiGCN_Twitter.py:45-56) and its weight gradient run as tiled masked products
                          instead of walks over each tree's list of positive root columns; needs a dense x.  Same
                          forward sums in the same order either way; 0 suits bag-of-words roots */
  int32_t edge_grad;   /* edge-weighted batch: 1 = features_backward keeps what bigcn_features_edge_grad reads (the
                          workspace must be bigcn_features_edge_workspace_bytes(dims, 1) bytes), with or without a
                          prepared buffer; 0 otherwise */
} bigcn_opts_t;

const char* bigcn_last_error(void);
int bigcn_join_internal_streams(bigcn_stream_t stream);
void* bigcn_internal_stream(void);
int bigcn_version(void);
/* 1 if the library carries sm_100a code and the current device is cc 10.x */
int bigcn_device_ok(void);

/* ---- graph prep ---------------------------------------------------------
 * Replaces gcn_norm / add_remaining_self_loops [torch_geometric], reached 4x
 * per forward from conv1/conv2 (BiGCN_Twitter.py:42,56,92,105), and the
 * Python max(data.batch) (:47) -- B is an argument, node_ptr comes from the
 * sorted batch vector.  Bit-exact vs oracle.gcn_oracle.graph_prep.
 * n_dirs = 1 or 2; edge_index[d] is [2,E[d]] int64; graphs[d] receives the
 * structure.  batch/node_ptr may be NULL (GCNConv called on its own). */
size_t bigcn_graph_prep_workspace_bytes(int64_t N, int64_t E_max, int32_t n_dirs);
/* Hub rows: a CSR row with more than BIGCN_LONG_ROW entries (the root of a reply tree in the
 * child-sum direction) is summed in fixed chunks by several half-warps and combined in chunk
 * order (deterministic, no atomics on floats).  graph prep lists those rows in in_long/out_long
 * (device int32 buffers of this many elements for a list of E edges); NULL = every row is walked
 * sequentially by its owner, in exact COO' order. */
#define BIGCN_LONG_ROW 32
size_t bigcn_long_ws_ints(int64_t E);
int bigcn_graph_prep(int32_t n_dirs, const int64_t* const* edge_index, const int64_t* E,
                     int64_t N, const int64_t* batch, int64_t B, int32_t deg_by,
                     const bigcn_graph_t* graphs, int32_t* node_ptr /*[B+1] or NULL*/,
                     int32_t* flags, void* workspace, size_t workspace_bytes,
                     bigcn_stream_t stream);

/* ---- X * W^T ------------------------------------------------------------
 * Replaces GCNConv.lin (cuBLAS SGEMM) at BiGCN_Twitter.py:42,92.
 * y[N, 64*n_w] = x[N,K] * [w0; w1]^T with w0, w1 the [64,K] lin.weight tensors (row pitch
 * ldw) of one or two directions (w1 = NULL for one), so TD and BU share ONE pass over x.
 * gemm_mode FP32: exact-fp32 streaming scan; TF32 / TF32X3: tcgen05 + TMA + TMEM GEMM; BF16: x holds bf16
 * rows (pitch K), tcgen05 kind::f16 with the weights split into bf16 terms.
 * scratch: bigcn_xw_scratch_floats(K, n_w) floats.  ldy = row pitch of y. */
size_t bigcn_xw_scratch_floats(int64_t K, int32_t n_w);
int bigcn_xw(const float* x, int64_t N, int64_t K, const float* w0, const float* w1, int64_t ldw,
             float* y, int64_t ldy, int32_t gemm_mode, float* scratch, bigcn_stream_t stream);
/* The autograd transpose of the above (dW1 = T1^T X, SURVEY.md appendix B):
 * dw_d[o, k] = sum_i t[i, 64*d + o] * x[i, k] for d < n_w; t is [N, 64*n_w] dense.
 * FP32: exact streaming scan; TF32: one tcgen05 pass; TF32X2 / MIXED: T split hi + lo (fp32-class only when x is
 * TF32-representable); TF32X3: T and x split; BF16: x holds bf16 rows, kind::f16 with t split into bf16 terms.
 * N = 0 writes zeros (x and t may then be NULL). */
size_t bigcn_xw_wgrad_scratch_floats(int64_t N, int64_t K, int32_t n_w);
int bigcn_xw_wgrad(const float* x, int64_t N, int64_t K, const float* t, int32_t n_w, float* dw0,
                   float* dw1, int64_t ldw, int32_t gemm_mode, float* scratch, bigcn_stream_t stream);
/* The input gradient of the above, same kernel as bigcn_features_x_grad:
 * dx[i, k] = sum_{d < n_w} sum_o t[i, 64*d + o] * w_d[o, k]; t is [N, 64*n_w] dense, w0 / w1 the [64,K] weights
 * (row pitch ldw; w1 = NULL for one).  Exactly one of dx (fp32) / dx_bf16 (bf16) is non-NULL, [N,K] dense; any K >= 1.
 * scratch: bigcn_x_dgrad_scratch_floats(N, K, n_w) floats, 16 B aligned. */
size_t bigcn_x_dgrad_scratch_floats(int64_t N, int64_t K, int32_t n_w);
int bigcn_x_dgrad(const float* t, int32_t n_w, const float* w0, const float* w1, int64_t ldw, int64_t N, int64_t K,
                  float* dx, void* dx_bf16, float* scratch, bigcn_stream_t stream);
/* The same input gradient for a CSR x (ptr [N+1], col [nnz], int32), sampled at x's stored entries (an SDDMM, the
 * convention of torch.sparse.mm's gradient): for every entry e < ptr[N] of row i,
 *   dval[e] = sum_{d < n_w} sum_o t[i, 64*d + o] * w_d[o, col[e]]
 * in plain fp32 FMAs (no TF32), deterministic (no atomics).  Every stored entry gets its value: explicit zeros, and
 * each duplicate (row, col) entry in full.  An entry whose column is outside [0, K) gets 0 (the forward skips it).
 * nnz is the length of dval: the entries in [ptr[N], nnz) are set to 0 (a CSR handed over at capacity), and
 * nothing at or past nnz is read or written.  t is [N, 64*n_w] dense, 16 B aligned; w0 / w1 as above.
 * scratch (W transposed): bigcn_x_dgrad_csr_scratch_floats(K, n_w) floats, 16 B aligned. */
size_t bigcn_x_dgrad_csr_scratch_floats(int64_t K, int32_t n_w);
int bigcn_x_dgrad_csr(const int32_t* ptr, const int32_t* col, int64_t N, int64_t K, int64_t nnz, const float* t,
                      int32_t n_w, const float* w0, const float* w1, int64_t ldw, float* dval, float* scratch,
                      bigcn_stream_t stream);
/* The same product and gradient through the row-sparse view of x (BIGCN_GEMM_SPARSE, for
 * bag-of-words inputs: Process/getTwittergraph.py:16-24 densifies `index:count` pairs).
 * bigcn_xw_sparse: exact fp32 scan that also records the non-zeros of x, then CSR
 * (ptr,col,val) and, through a stable radix sort, the column-sorted CSC (cptr,crow,cval) in
 * the workspace.  bigcn_xw_wgrad_sparse: dw_d[o,k] = sum over column k of x (rows ascending) of
 * x[i,k] * t[i, 64 d + o] -- no second pass over x; NaN (and BIGCN_FLAG_X_NOT_SPARSE raised by
 * the forward) when x holds more than N*min(K,48) non-zeros.  state[0] = nnz. */
size_t bigcn_xsparse_workspace_bytes(int64_t N, int64_t K);
int bigcn_xw_sparse(const float* x, int64_t N, int64_t K, const float* w0, const float* w1, int64_t ldw,
                    float* y, int64_t ldy, int32_t build_csc /* 0: product only (inference) */,
                    int32_t* flags, void* workspace, size_t workspace_bytes, bigcn_stream_t stream);
/* The pass over x that bigcn_batch_prepare runs a step ahead, on its own: captures the non-zeros of every row into
 * the ELL slots of a bigcn_xw_sparse workspace (no product); build_csr != 0 adds the scan + compaction into CSR. */
int bigcn_x_capture(const float* x, int64_t N, int64_t K, int32_t build_csr, int32_t* flags, void* workspace,
                    size_t workspace_bytes, bigcn_stream_t stream);
int bigcn_xw_wgrad_sparse(int64_t N, int64_t K, const float* t, int32_t n_w, float* dw0, float* dw1,
                          int64_t ldw, void* workspace, size_t workspace_bytes, bigcn_stream_t stream);
int bigcn_xsparse_view(int64_t N, int64_t K, void* workspace, size_t workspace_bytes, int32_t** state,
                       int32_t** ptr, int32_t** col, float** val, int32_t** cptr, int32_t** crow,
                       float** cval);
/* HOST function: one pass over a dense row-major host matrix (pinned or pageable) with
 * n_threads host threads (0 = all cores) that keeps the non-zero entries as CSR in host
 * buffers, columns ascending in every row -- 8 bytes per non-zero cross PCIe instead of
 * 4*K bytes per row.  No arithmetic.  Returns nnz, or -(needed nnz) when cap is too small. */
int64_t bigcn_host_dense_to_csr(const float* x, int64_t N, int64_t K, int32_t* ptr /*[N+1]*/,
                                int32_t* col /*[cap]*/, float* val /*[cap]*/, int64_t cap,
                                int32_t n_threads);
/* STREAM-style probe of the host-memory read bandwidth the compaction threads get (GB/s); data movement only. */
double bigcn_host_read_gbs(const void* buf, int64_t bytes, int32_t n_threads, int32_t reps);
/* wt[k, col0+o] = w[o, k0+k] for o<64: lays PyG [out,in] weights out for bigcn_xw */
int bigcn_transpose_weight(const float* w, int64_t ldw, int64_t k0, int64_t K,
                           float* wt, int64_t ldwt, int64_t col0, bigcn_stream_t stream);

/* ---- propagate ----------------------------------------------------------
 * Replaces MessagePassing.propagate + bias [torch_geometric] (index_select,
 * broadcast mul, atomic scatter_add) inside every GCNConv call.
 * out[i] = sum_{e in ptr[i]..ptr[i+1]} (dis[idx[e]]*dis[i]) * h[idx[e]]
 *          + (dis[i]*dis[i]) * h[i]  (+ bias) (relu)
 * summed in COO' order, no atomics, deterministic.  Pass in_ptr/in_idx for
 * A-hat, out_ptr/out_idx for A-hat^T (backward).  ldh, ldo multiples of 4, 16 B aligned rows. */
int bigcn_propagate(const int32_t* ptr, const int32_t* idx, const float* dis, int64_t N, int64_t E,
                    int32_t* long_ws /* in_long / out_long of that CSR, or NULL */,
                    const float* h, int64_t ldh, const float* bias /*or NULL*/, int32_t relu,
                    float* out, int64_t ldo, bigcn_stream_t stream);

/* ---- readout ------------------------------------------------------------
 * Replaces the second root-extend loop + torch_scatter.scatter_mean(x, data.batch, dim=0)
 * (BiGCN_Twitter.py:58-65) of one direction:
 *   feat[b, f]      = mean_{i in tree b} h2[i, f]          f < 64
 *   feat[b, 64 + f] = h1[rootindex[b], f]                  (mean of n_b copies of the root row)
 * node_ptr[B+1] comes from graph prep; trees of any size (slices of 512 rows are summed by
 * separate CTAs and combined in slice order: deterministic).  pos (or NULL) receives
 * #{i in tree b : h2[i,f] > 0}, which the backward uses for db2.  feat row pitch ldfeat. */
size_t bigcn_readout_scratch_floats(int64_t N, int64_t B);
int bigcn_readout(const float* h2 /*[N,64]*/, const float* h1 /*[N,64]*/, const int32_t* node_ptr,
                  const int64_t* rootindex, int64_t N, int64_t B, float* feat, int64_t ldfeat,
                  float* pos /*[B,64] or NULL*/, float* scratch, int32_t* flags, bigcn_stream_t stream);

/* scatter_mean backward on its own: grad_h2[i, :] = grad_feat[batch[i], 0:64] / n_b (the h1[root] half of
 * feat carries no gradient: copy.copy at BiGCN_Twitter.py:44 detaches it).  The fused training path
 * (bigcn_features_backward) forms this inside its gather instead. */
int bigcn_readout_backward(const float* grad_feat /*[B,ldg]*/, int64_t ldg, const int32_t* node_ptr,
                           const int64_t* batch, int64_t N, int64_t B, float* grad_h2 /*[N,64]*/,
                           bigcn_stream_t stream);

/* out[f] = sum_i g[i, f] for a dense [N,64] matrix: the bias gradient of a propagate on its own
 * (fixed chunks, fixed combine order: deterministic). */
size_t bigcn_colsum64_scratch_floats(int64_t N);
int bigcn_colsum64(const float* g, int64_t N, float* out /*[64]*/, float* scratch, bigcn_stream_t stream);

/* ---- dropout mask spec (tests) -----------------------------------------
 * keep[i,c] (uint8) for c < n_cols of the concatenated [h1|root_extend] tensor
 * (BiGCN_Twitter.py:51-54); stream = 0 (TD) / 1 (BU). */
int bigcn_dropout_mask(uint64_t seed, int32_t stream_id, int64_t node_id_base, int64_t N,
                       int64_t n_cols, float p, uint8_t* keep, bigcn_stream_t stream);

/* ---- GCNConv on its own -------------------------------------------------
 * conv(x, edge_index) as called at explain_PHEME.py:95,132.  w is [64,K]
 * (lin.weight), bias [64]; out [N,64].  Backward returns dw, db (x is an input of the
 * path and carries no gradient, SURVEY.md appendix B).  gemm_mode BIGCN_GEMM_BF16: x holds bf16 rows (pitch K)
 * in both calls. */
size_t bigcn_gcnconv_workspace_bytes(int64_t N, int64_t E, int64_t K);
int bigcn_gcnconv_forward(const float* x, int64_t N, int64_t K, const int64_t* edge_index,
                          int64_t E, const float* w, const float* bias, int32_t deg_by,
                          int32_t gemm_mode, float* out, int32_t* flags, void* workspace,
                          size_t workspace_bytes, bigcn_stream_t stream);
int bigcn_gcnconv_backward(const float* x, int64_t N, int64_t K, int64_t E,
                           const float* grad_out /*[N,64]*/, float* dw /*[64,K]*/, float* db /*[64]*/,
                           int32_t gemm_mode, void* workspace /* the forward's */, size_t workspace_bytes,
                           bigcn_stream_t stream);

/* ---- edge-weighted GCNConv (SURVEY.md 8f N3) -----------------------------
 * conv(x, edge_index, edge_weight) as EBGCN calls it (model/Twitter/EBGCN.py:84,181:
 * `self.conv2(x, edge_index, edge_weight=edge_pred)`), and gcn_norm with weights as
 * explain_PHEME.py:62-63 calls it.  Semantics of torch_geometric's gcn_norm /
 * add_remaining_self_loops(fill_value = 1): a self-loop edge in the list hands its weight to the
 * node's loop (the last one wins), other nodes get a unit loop; deg = sum of weights at the target
 * (source for BIGCN_DEG_BY_SOURCE) in edge-list order, then the loop; dis = deg^-1/2, inf -> 0;
 * norm_e = (dis[row] * w_e) * dis[col].
 *   gcn_norm_weighted: norm_e [E] per edge of the list (0 for self-loop edges: their weight sits
 *   in norm_self), norm_self [N], dis [N].
 *   forward: out = A-hat_w (x W^T) + bias, summed per row in edge-list order (deterministic).
 *   backward: dw [64,K], db [64], and optionally d_edge_weight [E] (directly and through the
 *   degrees) and dx [N,K] = (A-hat_w^T grad_out) W; NULL skips either.  Takes the forward's
 *   workspace (it keeps x W^T and the normalised structure). */
size_t bigcn_gcn_norm_weighted_workspace_bytes(int64_t N, int64_t E);
int bigcn_gcn_norm_weighted(const int64_t* edge_index /*[2,E]*/, int64_t E, const float* edge_weight /*[E]*/,
                            int64_t N, int32_t deg_by, float* norm_e, float* norm_self, float* dis,
                            int32_t* flags, void* workspace, size_t workspace_bytes, bigcn_stream_t stream);
size_t bigcn_gcnconv_weighted_workspace_bytes(int64_t N, int64_t E, int64_t K);
int bigcn_gcnconv_weighted_forward(const float* x, int64_t N, int64_t K, const int64_t* edge_index, int64_t E,
                                   const float* edge_weight, const float* w, const float* bias,
                                   int32_t deg_by, int32_t gemm_mode, float* out, int32_t* flags,
                                   void* workspace, size_t workspace_bytes, bigcn_stream_t stream);
int bigcn_gcnconv_weighted_backward(const float* x, int64_t N, int64_t K, const int64_t* edge_index, int64_t E,
                                    const float* edge_weight, const float* w, const float* grad_out,
                                    float* dw, float* db, float* d_edge_weight /*[E] or NULL*/,
                                    float* dx /*[N,K] or NULL*/, int32_t deg_by, int32_t gemm_mode,
                                    void* workspace, size_t workspace_bytes, bigcn_stream_t stream);

/* ---- the two-direction feature path ------------------------------------
 * Replaces TDrumorGCN.forward / BUrumorGCN.forward (BiGCN_Twitter.py:26-67,
 * 77-114): conv1, root-extend, relu, dropout, conv2, relu, root-extend,
 * scatter_mean.  feat[B,256] = [BU mean(H2) | BU H1[root] | TD mean(H2) | TD H1[root]]
 * (the cat order of :128).  The workspace carries what backward needs. */
size_t bigcn_features_workspace_bytes(const bigcn_dims_t* dims);
int bigcn_features_forward(const bigcn_dims_t* dims, const bigcn_batch_t* batch,
                           const bigcn_params_t* params, const bigcn_opts_t* opts,
                           float* feat /*[B,256]*/, int32_t* flags, void* workspace,
                           size_t workspace_bytes, bigcn_stream_t stream);
/* The weight-independent half of a step, one step AHEAD: graph structure of both directions, node pointers, the root
 * rows' positive columns and (BIGCN_GEMM_SPARSE) the non-zeros of x as CSR + column-sorted CSC, written into
 * `prepared` (bigcn_batch_prepare_bytes(dims) bytes) on two lowest-priority internal streams that fork from
 * `stream` at the call.  Call it for batch i+1 right before enqueuing step i and bigcn_batch_prepare_join(stream)
 * right after step i: the HBM-bound pass over the next x then overlaps the latency-bound kernels of the current
 * step (the role of the reference's DataLoader worker processes, BiGCN_Twitter.py:168).  Capturable: fork and join
 * sit on `stream`.  Then pass the buffer as batch->prepared to the three calls of step i+1.  An edge-weighted batch
 * (td_edge_weight / bu_edge_weight set) also gets the weighted normalisation of the directions opts.dir_mask selects
 * (graph prep with the edge ids, loop weights, weighted degrees, normalised weights in both CSR orders), written after
 * the unweighted layout: its buffer is bigcn_batch_prepare_edge_bytes(dims) bytes, and the weighted step no longer
 * computes any of it.  A non-finite weight or a negative weighted degree raises BIGCN_FLAG_EDGE_WEIGHT in `flags`. */
size_t bigcn_batch_prepare_bytes(const bigcn_dims_t* dims);
size_t bigcn_batch_prepare_edge_bytes(const bigcn_dims_t* dims);
int bigcn_batch_prepare(const bigcn_dims_t* dims, const bigcn_batch_t* batch, const bigcn_opts_t* opts, int32_t* flags,
                        void* prepared, size_t prepared_bytes, bigcn_stream_t stream);
int bigcn_batch_prepare_join(bigcn_stream_t stream);
/* grad_feat[B,256] -> gradients of the eight conv tensors (fc_* untouched).
 * The gradient through the second root-extend is dropped, as copy.copy does at :44. */
int bigcn_features_backward(const bigcn_dims_t* dims, const bigcn_batch_t* batch,
                            const bigcn_params_t* params, const bigcn_opts_t* opts,
                            const float* grad_feat, const bigcn_params_t* grads,
                            void* workspace, size_t workspace_bytes, bigcn_stream_t stream);
/* Workspace of the three calls above for a batch with td_edge_weight / bu_edge_weight: the unweighted workspace, then
 * the weighted normalisation of both directions; edge_grad = 1 adds room for the products the edge gradient reads
 * (4 * N * 64 floats more: backward then writes T2 and G1 beside X W1^T and conv2's input instead of over them). */
size_t bigcn_features_edge_workspace_bytes(const bigcn_dims_t* dims, int32_t edge_grad);
/* Gradient w.r.t. the edge weights: d_td_w [E_td] / d_bu_w [E_bu] (either may be NULL; the batch must carry that
 * direction's weights).  Call after bigcn_features_backward with the same dims, batch, opts (edge_grad = 1) and
 * workspace.  Per direction it sums over conv1 and conv2 dL/dnorm_e = <G1[c], XW[r]> + <G2[c], M[r]> (taken by the
 * backward) and carries it through the normalisation: dis_r dis_c dL/dnorm_e + dL/ddeg of the degree node; a self-loop
 * edge of the list gets its node's loop gradient (every such edge, as autograd of the reference's index_put gives).
 * A prepared batch (batch->prepared) reads the normalisation from that buffer, the products from the workspace.
 * The chain forks onto the library's low-priority stream from the point right after the backward's per-edge products,
 * so it runs underneath the backward's last propagate and dW1, and joins `stream` before returning; do not enqueue
 * another features_backward between the two calls.  Deterministic, no floating-point atomics. */
int bigcn_features_edge_grad(const bigcn_dims_t* dims, const bigcn_batch_t* batch, const bigcn_opts_t* opts,
                             float* d_td_w, float* d_bu_w, void* workspace, size_t workspace_bytes,
                             bigcn_stream_t stream);
/* Gradient w.r.t. data.x (dense x): the reference's conv1 reads x (BiGCN_Twitter.py:42) while its root-extend reads
 * the detached copy.copy x1 (:28,45-50), so only conv1 carries one back: dX = sum over the directions of T1_d W1_d
 * with T1_d = A-hat_d^T G1_d, the matrix whose transpose product is dW1.  Call after bigcn_features_backward with the
 * same dims, params, opts and workspace (it reads T1 from there; dir_mask selects the directions).
 * Exactly one of dx (fp32 [N,K]) and dx_bf16 (bf16 [N,K], each element rounded once to nearest even) is non-NULL.
 * tcgen05 kind::tf32 in the 3xTF32 form (T_hi W_hi + T_hi W_lo + T_lo W_hi): fp32-class; deterministic (no atomics).
 * scratch: bigcn_x_dgrad_scratch_floats(N, K, n_w) floats, 16 B aligned. */
int bigcn_features_x_grad(const bigcn_dims_t* dims, const bigcn_params_t* params, const bigcn_opts_t* opts,
                          float* dx, void* dx_bf16, float* scratch, void* workspace, size_t workspace_bytes,
                          bigcn_stream_t stream);
/* Gradient w.r.t. a CSR data.x (batch->x = NULL, x_ptr / x_col / x_val, gemm_mode BIGCN_GEMM_SPARSE): the dX above
 * sampled at x's stored entries, dval[e] = (T1cat[i] . W1cat^T[col[e]]) for entry e of row i -- the gradient of
 * x_val.  Same kernel and conventions as bigcn_x_dgrad_csr (nnz = the length of dval; [ptr[N], nnz) set to 0).
 * Call after bigcn_features_backward with the same dims, batch, opts and workspace: it reads T1cat, and W1^T as
 * bigcn_features_forward laid it out, from there (dir_mask selects the directions); no scratch. */
int bigcn_features_x_grad_csr(const bigcn_dims_t* dims, const bigcn_batch_t* batch, const bigcn_opts_t* opts,
                              float* dval, int64_t nnz, void* workspace, size_t workspace_bytes,
                              bigcn_stream_t stream);

/* ---- head ---------------------------------------------------------------
 * Replaces fc + log_softmax (BiGCN_Twitter.py:129-130). */
int bigcn_head_forward(const float* feat, int64_t B, int64_t C, const float* fc_w,
                       const float* fc_b, float* logp /*[B,C]*/, bigcn_stream_t stream);
size_t bigcn_head_backward_scratch_floats(int64_t B, int64_t C);
int bigcn_head_backward(const float* grad_logp, const float* logp, const float* feat, int64_t B,
                        int64_t C, const float* fc_w, float* grad_feat /*[B,256]*/,
                        float* d_fc_w, float* d_fc_b, float* scratch, size_t scratch_floats,
                        bigcn_stream_t stream);

/* The training step's head in one call: bigcn_head_forward + bigcn_nll_loss + bigcn_head_backward
 * (same arithmetic).  One launch on `stream` produces logp and grad_feat; d_fc_w, d_fc_b and the
 * loss scalar are finished on the library's side stream and are ordered before whatever
 * bigcn_features_backward / bigcn_adam_step / bigcn_dp_reduce_adam later do on `stream`. */
size_t bigcn_head_train_scratch_floats(int64_t B, int64_t C);
int bigcn_head_train(const float* feat, const int64_t* y, int64_t B, int64_t C, int64_t B_global,
                     const float* fc_w, const float* fc_b, float* logp, float* loss, float* grad_feat,
                     float* d_fc_w, float* d_fc_b, float* scratch, size_t scratch_floats,
                     bigcn_stream_t stream);

/* The training step's tail in ONE launch on `stream`: the readout's second pass (feat), bigcn_head_train's
 * arithmetic (logp, loss, grad_feat, fc gradients on the side stream) and the scatter_mean backward's
 * per-tree scaling that bigcn_features_backward starts with.  Call order, all with opts.fused_tail = 1 and
 * the same dims / workspace: bigcn_features_forward -> bigcn_train_tail -> bigcn_features_backward.
 * scratch: bigcn_head_train_scratch_floats(B, C) floats. */
int bigcn_train_tail(const bigcn_dims_t* dims, const bigcn_batch_t* batch, const bigcn_opts_t* opts, float* feat,
                     const int64_t* y, int64_t B_global, const float* fc_w, const float* fc_b, float* logp,
                     float* loss, float* grad_feat, float* d_fc_w, float* d_fc_b, float* scratch,
                     size_t scratch_floats, int32_t* flags, void* workspace, size_t workspace_bytes,
                     bigcn_stream_t stream);

/* Evaluation bookkeeping on the device (SURVEY.md 8f N4): adds this batch to
 * counts[C][4] = {TP, FN, FP, TN} per class and totals[3] = {trees, correct, sum(-logp[y]) * 1e6}
 * (int64, zero-initialised by the caller, accumulated over an epoch, read back once).  Replaces
 * out.max(dim=-1) + tools/evaluate.py:3-31 / :93-108 and the per-batch .item() syncs of
 * BiGCN_Twitter.py:188-191,217-225. */
int bigcn_eval_counts(const float* logp, const int64_t* y, int64_t B, int64_t C, int64_t* counts,
                      int64_t* totals, bigcn_stream_t stream);

/* ---- loss and optimiser (the step around the path, :184-189, :146-153) --
 * loss = -(1/B_global) sum_b logp[b,y[b]] (F.nll_loss, mean); grad_logp = dloss/dlogp. */
int bigcn_nll_loss(const float* logp, const int64_t* y, int64_t B, int64_t C, int64_t B_global,
                   float* loss /*[1]*/, float* grad_logp /*[B,C] or NULL*/, bigcn_stream_t stream);
/* torch.optim.Adam (coupled L2) over one flat buffer; lr_of_segment: n_seg pairs
 * (end_offset, lr) on the DEVICE; step_count: device int64[4], zero-initialised by the caller:
 * [0] the step, advanced here by the last block of the update kernel, [1] its arrival counter,
 * [2] calls counter (advanced with [0]; never rewound by a checkpoint load): what opts.seed_dev points
 * at so that every step -- eager or a CUDA-graph replay -- draws a fresh dropout mask, [3] arrival counter of the
 * push phase of bigcn_dp_reduce_adam. */
int bigcn_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq,
                    int64_t n, const int64_t* seg_end, const float* seg_lr, int32_t n_seg,
                    double beta1, double beta2, double eps, double weight_decay,
                    double grad_scale, int64_t* step_count, bigcn_stream_t stream);

/* ---- dense rows -> CSR on the device (the device half of bigcn_b200.HostFeeder) ------------------
 * The reference's loader hands over DENSE bag-of-words rows (Process/dataset.py:64-99).  A feeder
 * sends part of a batch's rows over PCIe as they are while the host compacts the rest
 * (bigcn_host_dense_to_csr); these two calls turn the dense part into CSR entries that continue the
 * host part's arrays.  dense_row_counts: non-zeros per row.  The caller forms the inclusive prefix
 * of the counts; dense_rows_to_csr then writes row r's entries (ascending columns) at
 * base + incl[r-1] and ptr_out[r] = base + incl[r] (ptr_out points at the combined row pointer's
 * entry of row 0 + 1).  Entries that would pass cap (the capacity of col / val) are dropped, the
 * row pointer stops growing and BIGCN_FLAG_X_NOT_SPARSE is set in *flags: never an out-of-bounds
 * write, never a silent wrong answer. */
int bigcn_dense_row_counts(const float* x, int64_t N, int64_t K, int32_t* cnt, bigcn_stream_t stream);
/* The same count for a bf16 x [N,K] (row pitch K): the density probe of BIGCN_GEMM_BF16 (dense or bag-of-words rows). */
int bigcn_dense_row_counts_bf16(const void* x, int64_t N, int64_t K, int32_t* cnt, bigcn_stream_t stream);
int bigcn_dense_rows_to_csr(const float* x, int64_t N, int64_t K, const int32_t* incl_counts, int64_t base,
                            int32_t* ptr_out, int32_t* col, float* val, int64_t cap, int32_t* flags,
                            bigcn_stream_t stream);

/* ---- on-device batch assembly + DropEdge (SURVEY.md 8f N2) --------------------------------------
 * For a dataset packed in HBM (all trees: node_ptr/edge_ptr [T+1], local edge lists, x as CSR over
 * all nodes, local root index, label) builds the batch of trees tree_id[0..B): what
 * BiGraphDataset.__getitem__ (Process/dataset.py:64-99: DropEdge keeps int(e*(1-rate)) positions of
 * the TD and, independently, of the BU list, order preserved) and PyG's collate
 * (BiGCN_Twitter.py:168: concatenate, offset the *index keys by the node count, batch vector) do on
 * the host.  The caller computes the four offset arrays on the host from the tree sizes
 * (td_off/bu_off: kept edges per tree) -- no synchronisation; tree_id and the four offset arrays [B+1]
 * may be device memory or PINNED HOST memory the kernels read in place (then the caller must not rewrite
 * them before the launches have completed).  Outputs: the five attributes
 * forward(data) reads, with data.x as CSR (ox_ptr/ox_col/ox_val), and y. */
int bigcn_assemble_batch(const int64_t* node_ptr, const int64_t* edge_ptr, const int32_t* edge_src,
                         const int32_t* edge_dst, const int64_t* x_ptr, const int32_t* x_col,
                         const float* x_val, const int32_t* root_local, const int64_t* y_all,
                         const int64_t* tree_id, const int64_t* node_off, const int64_t* td_off,
                         const int64_t* bu_off, const int64_t* nnz_off, int64_t B, int64_t E_td,
                         int64_t E_bu, uint64_t seed, int64_t* edge_index, int64_t* bu_edge_index,
                         int64_t* batch, int64_t* rootindex, int64_t* y, int32_t* ox_ptr, int32_t* ox_col,
                         float* ox_val, bigcn_stream_t stream);
/* The same batch from a dataset whose features are DENSE rows: x_all [N_all, K] of elem_bytes = 4 (fp32) or 2 (bf16)
 * per element, row pitch K.  The same tree, edge and offset arguments and the same pinned-memory rule as
 * bigcn_assemble_batch (no x_ptr / x_col / x_val / nnz_off); ox [N, K] of the same element type receives tree
 * tree_id[b]'s rows at row node_off[b], copied bit for bit (no conversion).  16-byte loads and stores when K * elem_bytes
 * and both addresses are multiples of 16.  B = 0 returns 0; K < 1, K * elem_bytes >= 2^30, another elem_bytes or an
 * x_all / ox not aligned to elem_bytes fail. */
int bigcn_assemble_batch_dense(const int64_t* node_ptr, const int64_t* edge_ptr, const int32_t* edge_src,
                               const int32_t* edge_dst, const int32_t* root_local, const int64_t* y_all,
                               const int64_t* tree_id, const int64_t* node_off, const int64_t* td_off,
                               const int64_t* bu_off, int64_t B, int64_t E_td, int64_t E_bu, uint64_t seed,
                               int64_t* edge_index, int64_t* bu_edge_index, int64_t* batch, int64_t* rootindex,
                               int64_t* y, const void* x_all, int64_t K, int32_t elem_bytes, void* ox,
                               bigcn_stream_t stream);
/* Edge weights through the same assembly: every kept edge's weight lands at the position its edge takes in
 * edge_index / bu_edge_index (each direction after its own DropEdge subset, in kept order), copied bit for bit in the
 * launch that places the edges.  td_weight is one weight per tree edge, aligned with edge_src / edge_dst; bu_weight the
 * same for the BU list (NULL = td_weight: a reply carries one weight seen from either end). */
typedef struct bigcn_asm_weights {
  const float* td_weight;   /* [E_all]                             */
  const float* bu_weight;   /* [E_all] or NULL (= td_weight)       */
  float* edge_weight;       /* [E_td] out, aligned with edge_index */
  float* bu_edge_weight;    /* [E_bu] out, aligned with bu_edge_index */
} bigcn_asm_weights_t;
/* bigcn_assemble_batch / bigcn_assemble_batch_dense with weights (non-NULL); the same edges, nodes and features. */
int bigcn_assemble_batch_weighted(const int64_t* node_ptr, const int64_t* edge_ptr, const int32_t* edge_src,
                                  const int32_t* edge_dst, const int64_t* x_ptr, const int32_t* x_col,
                                  const float* x_val, const int32_t* root_local, const int64_t* y_all,
                                  const int64_t* tree_id, const int64_t* node_off, const int64_t* td_off,
                                  const int64_t* bu_off, const int64_t* nnz_off, int64_t B, int64_t E_td,
                                  int64_t E_bu, uint64_t seed, int64_t* edge_index, int64_t* bu_edge_index,
                                  int64_t* batch, int64_t* rootindex, int64_t* y, int32_t* ox_ptr, int32_t* ox_col,
                                  float* ox_val, const bigcn_asm_weights_t* weights, bigcn_stream_t stream);
int bigcn_assemble_batch_dense_weighted(const int64_t* node_ptr, const int64_t* edge_ptr, const int32_t* edge_src,
                                        const int32_t* edge_dst, const int32_t* root_local, const int64_t* y_all,
                                        const int64_t* tree_id, const int64_t* node_off, const int64_t* td_off,
                                        const int64_t* bu_off, int64_t B, int64_t E_td, int64_t E_bu, uint64_t seed,
                                        int64_t* edge_index, int64_t* bu_edge_index, int64_t* batch,
                                        int64_t* rootindex, int64_t* y, const void* x_all, int64_t K,
                                        int32_t elem_bytes, void* ox, const bigcn_asm_weights_t* weights,
                                        bigcn_stream_t stream);

/* ---- data-parallel optimiser step over peer memory (SURVEY.md 8e) -----------------------------
 * One kernel instead of "NCCL all-reduce of the flat gradient + Adam on every rank": grads[q] /
 * params[q] are rank q's flat buffers mapped into this process (symmetric memory over NVLink /
 * NVSwitch; HOST arrays of `world` device pointers).  This rank reduces the slice
 * bigcn_dp_slice(n, world, rank) of all ranks' gradients in rank order through peer loads, runs
 * Adam on its shard of exp_avg / exp_avg_sq (full-length local arrays, only the slice is used)
 * and stores the new parameters into every rank's buffer.  signals == NULL: the caller puts a cross-rank
 * barrier before (all gradients written) and after (all parameters written, gradients free again).
 * signals != NULL: HOST array of `world` device pointers, signals[q] = rank q's signal block in symmetric memory
 * (64 uint64, zero-initialised once; [32..35] receive globaltimer stamps of the last launch): both barriers then happen INSIDE the kernel (st.release.sys of an epoch
 * into every peer's block, ld.acquire.sys spins on the local one) -- one launch per step instead of three.
 * stage != NULL (needs signals): HOST array of `world` device pointers, stage[q] = rank q's staging buffer in symmetric
 * memory, world * bigcn_dp_stage_chunk(n, world) floats: every rank first PUSHES its gradient slices to their owners
 * (peer stores, one way) and then reduces its own slice from local memory -- no peer loads (NVLink round trips).
 * step_count[3] is that phase's arrival counter. */
int64_t bigcn_dp_stage_chunk(int64_t n, int32_t world);
int bigcn_dp_slice(int64_t n, int32_t world, int32_t rank, int64_t* lo, int64_t* hi);
int bigcn_dp_reduce_adam(const float* const* grads, float* const* params, int32_t world, int32_t rank,
                         float* exp_avg, float* exp_avg_sq, int64_t n, const int64_t* seg_end,
                         const float* seg_lr, int32_t n_seg, double beta1, double beta2, double eps,
                         double weight_decay, double grad_scale, int64_t* step_count,
                         void* const* signals, float* const* stage, bigcn_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* BIGCN_B200_H */
