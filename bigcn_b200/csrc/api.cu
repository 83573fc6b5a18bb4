// C-ABI orchestration: the two-direction feature path (forward / backward), GCNConv on its
// own, and the small exported helpers.  Every function only enqueues kernels on the caller's
// stream; the workspace carved here carries what backward needs.
#include <stdarg.h>
#include <stdlib.h>

#include "kernels.cuh"

namespace bigcn {

// ---- error / device helpers ---------------------------------------------------
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = 148;
  }
  return n;
}

// ---- side stream: short independent kernels run beside the long X stream -------------------
// One high-priority non-blocking stream and a few events per device, created on first use.
// Every entry point that forks onto it joins again before it returns, so at return all of its
// work is ordered on the caller's stream (and a CUDA-graph capture sees a fork/join diamond).
struct SideCtx {
  SideStream s;        // high priority: work the main stream will wait for soon (graph prep)
  cudaStream_t side2;  // high priority, a second short chain beside the first (root columns; dW2b)
  cudaStream_t low;    // lowest priority: work nobody waits for until much later (column sort of X)
  cudaStream_t prep[2];  // lowest priority: bigcn_batch_prepare of the NEXT batch, beside the whole current step
  cudaStream_t bw[2];    // lowest priority: the backward's dW2 / db chains -- nobody waits for them before the optimiser, so they
                         // must not take SM slots from G1 -> T1 -> dW1 (the caller's stream, see ops.step_stream) nor from this
                         // step's column sort, which the dW1 sweep waits for
  cudaEvent_t ev[16];
  bool ok;
};
static SideCtx* side_ctx() {
  static SideCtx ctx[64];
  static bool init[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  if (!init[dev]) {
    init[dev] = true;
    SideCtx& c = ctx[dev];
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);
    // four levels when the device has them (B200: 0 .. -3, lower = more urgent):
    //   hi      side / side2   short chains the main chain is about to wait for (graph prep inline, root columns)
    //   lo - 2  [the caller's step stream: bigcn_b200.ops.step_stream]
    //   lo - 1  low            this step's column sort of x: the dW1 sweep at the end of the chain waits for it
    //   lo      prep / bw      the NEXT batch's preparation; this step's dW2 / db chains (only the optimiser waits for them)
    const int mid = lo - 1 < hi ? hi : lo - 1;
    c.ok = cudaStreamCreateWithPriority(&c.s.side, cudaStreamNonBlocking, hi) == cudaSuccess &&
           cudaStreamCreateWithPriority(&c.side2, cudaStreamNonBlocking, hi) == cudaSuccess &&
           cudaStreamCreateWithPriority(&c.low, cudaStreamNonBlocking, mid) == cudaSuccess &&
           cudaStreamCreateWithPriority(&c.prep[0], cudaStreamNonBlocking, lo) == cudaSuccess &&
           cudaStreamCreateWithPriority(&c.prep[1], cudaStreamNonBlocking, lo) == cudaSuccess &&
           cudaStreamCreateWithPriority(&c.bw[0], cudaStreamNonBlocking, lo) == cudaSuccess &&
           cudaStreamCreateWithPriority(&c.bw[1], cudaStreamNonBlocking, lo) == cudaSuccess;
    for (int i = 0; i < 16 && c.ok; ++i) c.ok = cudaEventCreateWithFlags(&c.ev[i], cudaEventDisableTiming) == cudaSuccess;
    const char* e = getenv("BIGCN_NO_SIDE_STREAM");
    if (e && e[0] == '1') c.ok = false;
  }
  return ctx[dev].ok ? &ctx[dev] : nullptr;
}
// `to` waits for everything queued on `from` so far
static void stream_after(SideCtx* c, int ev, cudaStream_t from, cudaStream_t to) {
  cudaEventRecord(c->ev[ev], from);
  cudaStreamWaitEvent(to, c->ev[ev], 0);
}

// for the other translation units (head.cu): run something beside the caller's stream
cudaStream_t side_fork(cudaStream_t main_st) {
  SideCtx* c = side_ctx();
  if (!c) return main_st;
  stream_after(c, 4, main_st, c->s.side);
  return c->s.side;
}
void side_join(cudaStream_t main_st) {   // main waits for everything queued on the side stream
  SideCtx* c = side_ctx();
  if (c) stream_after(c, 5, c->s.side, main_st);
}

// w[0..n_w): PyG [64, K] weights (row pitch ldw).  scratch: 2 * 64 * n_w * K floats -- the
// transposed copy the fp32 scan streams, or the TF32 hi/lo split of the tensor-core modes.
int xw_dispatch(const float* x, int64_t N, int64_t K, const float* const* w, int n_w, int64_t ldw,
                float* scratch, float* y, int64_t ldy, int mode, cudaStream_t st) {
  BIGCN_CHECK_ARG(n_w == 1 || n_w == 2, "xw: one or two weight matrices");
  const int n_out = H * n_w;
  if (mode == BIGCN_GEMM_SPARSE) mode = BIGCN_GEMM_FP32;   // on its own the product is the exact scan
  if (mode == BIGCN_GEMM_FP32 || mode == BIGCN_GEMM_MIXED) {
    TransposeJobs js{};
    for (int q = 0; q < n_w; ++q) js.job[js.n++] = TransposeJob{w[q], ldw, 0, K, scratch, n_out, q * H};
    if (int rc = transpose_jobs_launch(js, st)) return rc;
    return xw_fp32(x, N, K, scratch, n_out, y, ldy, st);
  }
  BIGCN_CHECK_ARG(mode == BIGCN_GEMM_TF32 || mode == BIGCN_GEMM_TF32X3 || mode == BIGCN_GEMM_TF32X2 || mode == BIGCN_GEMM_BF16,
                  "xw: unknown gemm_mode %d", mode);
  return xw_tc_weights(x, N, K, w, ldw, n_out, scratch, y, ldy, mode, st);
}

// ---- workspace of the feature path -----------------------------------------------
struct FeatWs {
  bigcn_graph_t g[2];       // [0] = TD, [1] = BU
  int32_t* node_ptr;
  float* w1T;               // [K][128]  (TD cols 0..63, BU cols 64..127) | hi/lo split [4][64][K]
  float* w2aT[2];           // [64][64]
  float* xw_part;           // split-K partials of the tcgen05 X * W on small batches
  float* w2bT[2];           // [K][64]
  int32_t* rnz_cnt; int32_t* rnz_col; float* rnz_val;
  float* P[2];              // [B][64]
  float* xw;                // [N][128]      (backward: T2[0], T2[1] as two [N][64] halves)
  float* h1[2];             // [N][64]
  float* a1[2];             // [N][64]
  float* z[2];              // [N][64]       (backward: G2 then G1)
  float* h2[2];             // [N][64]       (backward: T1cat [N][128] once G2 is formed)
  float* cs_part[2];        // [chunks][64]  column-sum partials of db2 (written by the tail, summed on the side stream)
  float* cs_part1[2];       // [chunks][64]  ... of db1 (k_bwd_mix): a buffer of its own -- the side stream may still be
                            //               reading the db2 partials when k_bwd_mix writes these
  float* op_part[2];        // [chunks][4096]
  float* dw_part;           // dW1 slab partials
  float* dP[2];             // [B][64]
  int32_t* slot;            // [K][B] slot of column k in tree b's root list, or -1
  int32_t* overflow;        // [0] some root row has more than DW2B_CAP positive columns; [1 + k] column k is
                            // positive in some root row
  float* pos[2];            // [B][64] #{i in tree : H2[i][f] > 0}
  float* gs[2];             // [B][64] grad_feat / n_b
  unsigned long long* keep[2];  // [N] bit t: root slot t of the node's tree survived dropout (train mode)
  float* S[2];              // [(blocks + B)][DW2B_CAP][64] masked T2 sums per (row block, tree, slot)
  float* rootR[2];          // [splits][N][64] column-split partials of the dense-root product (rootdense.cu), small batches
  float* ro_part;           // readout slice partials
  XSparse xs;               // row-sparse view of X (gemm_mode SPARSE)
  void* prep_ws; size_t prep_bytes;
  size_t total;
};

// The weight-independent part of a step's workspace: what bigcn_batch_prepare fills for a batch (one step ahead of
// the step that consumes it) -- or, without a prepared buffer, the tail of the features workspace that
// features_forward fills itself.
struct PrepWs {
  bigcn_graph_t g[2];
  int32_t* node_ptr;
  int32_t* rnz_cnt; int32_t* rnz_col; float* rnz_val;
  int32_t* slot; int32_t* overflow;
  XSparse xs;
  void* prep_ws; size_t prep_bytes;
  size_t total;
};
static PrepWs carve_prepared(const bigcn_dims_t* dm, void* ws, size_t bytes) {
  PrepWs w{};
  Carver c(ws, bytes);
  const int64_t N = dm->N, B = dm->B, K = dm->K;
  const int64_t E[2] = {dm->E_td, dm->E_bu};
  for (int d = 0; d < 2; ++d) {
    w.g[d].in_ptr = c.take<int32_t>(N + 1);
    w.g[d].out_ptr = c.take<int32_t>(N + 1);
    w.g[d].in_idx = c.take<int32_t>(E[d] > 0 ? E[d] : 1);
    w.g[d].out_idx = c.take<int32_t>(E[d] > 0 ? E[d] : 1);
    w.g[d].deg = c.take<int32_t>(N > 0 ? N : 1);
    w.g[d].dis = c.take<float>(N > 0 ? N : 1);
    w.g[d].rowsum = nullptr;
    w.g[d].in_long = c.take<int32_t>(long_ws_ints(E[d]));
    w.g[d].out_long = c.take<int32_t>(long_ws_ints(E[d]));
  }
  w.node_ptr = c.take<int32_t>(B + 1);
  w.rnz_cnt = c.take<int32_t>(B > 0 ? B : 1);
  w.rnz_col = c.take<int32_t>((size_t)(B > 0 ? B : 1) * K);
  w.rnz_val = c.take<float>((size_t)(B > 0 ? B : 1) * K);
  w.slot = c.take<int32_t>((size_t)(B > 0 ? B : 1) * K);
  w.overflow = c.take<int32_t>(1 + K);
  w.xs = xs_carve(c, N, K);
  const int64_t Emax = E[0] > E[1] ? E[0] : E[1];
  w.prep_bytes = graph_prep_ws_bytes(N, Emax, 2);
  w.prep_ws = c.take<char>(w.prep_bytes);
  w.total = align_up(c.off, 256);
  return w;
}

static FeatWs carve_features(const bigcn_dims_t* dm, void* ws, size_t bytes, void* prepared = nullptr) {
  FeatWs w{};
  Carver c(ws, bytes);
  const int64_t N = dm->N, B = dm->B, K = dm->K;
  w.w1T = c.take<float>((size_t)K * 256);   // fp32: [K][128] transposed; tensor-core modes: hi/lo split
  for (int d = 0; d < 2; ++d) {
    w.w2aT[d] = c.take<float>(H * H);
    w.w2bT[d] = c.take<float>((size_t)K * H);
  }
  w.xw_part = c.take<float>(xw_tc_partial_floats());
  const size_t nh = (size_t)(N > 0 ? N : 1) * H;
  for (int d = 0; d < 2; ++d) w.P[d] = c.take<float>((size_t)(B > 0 ? B : 1) * H);
  w.xw = c.take<float>(2 * nh);
  w.h1[0] = c.take<float>(2 * nh);   // one block: the backward's dW1 GEMM keeps the lo half of T1's TF32 split here
  w.h1[1] = w.h1[0] + nh;
  for (int d = 0; d < 2; ++d) w.a1[d] = c.take<float>(nh);
  w.z[0] = c.take<float>(2 * nh);
  w.z[1] = w.z[0] + nh;
  w.h2[0] = c.take<float>(2 * nh);
  w.h2[1] = w.h2[0] + nh;
  int csn = cs_chunks(N) > bm_chunks(N) ? cs_chunks(N) : bm_chunks(N);
  if (gs_chunks(B) > csn) csn = gs_chunks(B);
  for (int d = 0; d < 2; ++d) w.cs_part[d] = c.take<float>((size_t)csn * H);
  for (int d = 0; d < 2; ++d) w.cs_part1[d] = c.take<float>((size_t)csn * H);
  for (int d = 0; d < 2; ++d) w.op_part[d] = c.take<float>((size_t)op_chunks(N) * H * H);
  w.dw_part = c.take<float>(dw_partial_floats(N, K, 128));
  for (int d = 0; d < 2; ++d) w.dP[d] = c.take<float>((size_t)(B > 0 ? B : 1) * H);
  for (int d = 0; d < 2; ++d) w.pos[d] = c.take<float>((size_t)(B > 0 ? B : 1) * H);
  for (int d = 0; d < 2; ++d) w.gs[d] = c.take<float>((size_t)(B > 0 ? B : 1) * H);
  {   // sparse roots: masked T2 sums per (row block, tree, slot); dense roots (rootdense.cu): [segments][K][64] partials
    const size_t s_sparse = (size_t)(dw2b_blocks(N) + B) * DW2B_CAP * H, s_dense = (size_t)K * H;
    for (int d = 0; d < 2; ++d) w.S[d] = c.take<float>(s_sparse > s_dense ? s_sparse : s_dense);
  }
  for (int d = 0; d < 2; ++d) w.keep[d] = c.take<unsigned long long>((size_t)(N > 0 ? N : 1));
  {
    const int64_t rows = 8 * (N > 0 ? N : 1);
    for (int d = 0; d < 2; ++d) w.rootR[d] = c.take<float>((size_t)(rows < RD_CAP_ROWS ? rows : RD_CAP_ROWS) * H);
  }
  w.ro_part = c.take<float>(readout_scratch_floats(N, B, 2));
  // the weight-independent part: the caller's prepared buffer, or the tail of this workspace
  const size_t step_bytes = align_up(c.off, 256);
  char* tail = ws ? reinterpret_cast<char*>(ws) + step_bytes : nullptr;
  const PrepWs pw = carve_prepared(dm, prepared ? prepared : tail, 0);
  w.g[0] = pw.g[0]; w.g[1] = pw.g[1];
  w.node_ptr = pw.node_ptr;
  w.rnz_cnt = pw.rnz_cnt; w.rnz_col = pw.rnz_col; w.rnz_val = pw.rnz_val;
  w.slot = pw.slot; w.overflow = pw.overflow;
  w.xs = pw.xs;
  w.prep_ws = pw.prep_ws; w.prep_bytes = pw.prep_bytes;
  w.total = step_bytes + pw.total;   // sized for the self-contained case whether or not `prepared` is given
  return w;
}

// An edge-weighted batch: the weighted normalisation of both directions (weighted.cu), laid out after the features
// workspace; with opts.edge_grad also the buffers that keep XW and Z alive through the backward and the per-edge
// products of the edge gradient.
struct WFeatWs {
  WGraph G[2];
  float* in_w[2];           // [E] normalised weight per by-target entry (forward sweeps)
  float* out_w[2];          // [E] ... per by-source entry (A-hat^T sweeps)
  float* ones;              // [Emax] the weights of a direction the caller gave none
  float* t2;                // edge_grad: [2][N][64] T2, instead of over XW
  float* g1;                // edge_grad: [2][N][64] G1, instead of over Z
  float* a_e[2];            // edge_grad: [E] dL/dnorm per edge id
  float* a_self[2];         // edge_grad: [N] ... per self-loop
  float* ddeg[2];           // edge_grad: [N]
  size_t total;
};
static WFeatWs carve_wfeat(const bigcn_dims_t* dm, void* base, bool edge_grad) {
  WFeatWs w{};
  Carver c(base, 0);
  const int64_t N = dm->N;
  const int64_t E[2] = {dm->E_td, dm->E_bu};
  const size_t n1 = (size_t)(N > 0 ? N : 1);
  for (int d = 0; d < 2; ++d) {
    const size_t e1 = (size_t)(E[d] > 0 ? E[d] : 1);
    w.G[d].in_eid = c.take<int32_t>(e1);
    w.G[d].out_eid = c.take<int32_t>(e1);
    w.G[d].loop_eid = c.take<int32_t>(n1);
    w.G[d].self_w = c.take<float>(n1);
    w.G[d].dis = c.take<float>(n1);
    w.G[d].norm_e = c.take<float>(e1);
    w.G[d].norm_self = c.take<float>(n1);
    w.in_w[d] = c.take<float>(e1);
    w.out_w[d] = c.take<float>(e1);
  }
  w.ones = c.take<float>((size_t)(E[0] > E[1] ? E[0] : E[1]) + 1);
  if (edge_grad) {
    w.t2 = c.take<float>(2 * n1 * H);
    w.g1 = c.take<float>(2 * n1 * H);
    for (int d = 0; d < 2; ++d) {
      w.a_e[d] = c.take<float>((size_t)(E[d] > 0 ? E[d] : 1));
      w.a_self[d] = c.take<float>(n1);
      w.ddeg[d] = c.take<float>(n1);
    }
  }
  w.total = align_up(c.off, 256);
  return w;
}
static bool batch_weighted(const bigcn_batch_t* bt) { return bt->td_edge_weight != nullptr || bt->bu_edge_weight != nullptr; }
static const float* dir_edge_weight(const bigcn_batch_t* bt, int d) { return d == 0 ? bt->td_edge_weight : bt->bu_edge_weight; }
// A weighted batch prepared ahead: bigcn_batch_prepare writes the normalisation right after the unweighted layout
static WFeatWs carve_prepared_wfeat(const bigcn_dims_t* dm, void* prepared) {
  const size_t base = carve_prepared(dm, nullptr, 0).total;
  return carve_wfeat(dm, prepared ? reinterpret_cast<char*>(prepared) + base : nullptr, false);
}
// The weighted section a step reads: the workspace's own (features_forward fills it), with the normalisation taken from
// the prepared buffer instead when the batch came prepared (the edge-gradient buffers stay in the workspace)
static WFeatWs step_wfeat(const bigcn_dims_t* dm, const bigcn_batch_t* bt, void* ws, size_t feat_total, bool edge_grad) {
  WFeatWs wf = carve_wfeat(dm, ws ? reinterpret_cast<char*>(ws) + feat_total : nullptr, edge_grad);
  if (bt->prepared != nullptr) {
    const WFeatWs pw = carve_prepared_wfeat(dm, bt->prepared);
    for (int d = 0; d < 2; ++d) {
      wf.G[d] = pw.G[d];
      wf.in_w[d] = pw.in_w[d];
      wf.out_w[d] = pw.out_w[d];
    }
    wf.ones = pw.ones;
  }
  return wf;
}
// the weighted normalisation of the active directions on top of graph prep (a direction without weights: all ones)
static int wfeat_prep_dirs(const bigcn_dims_t* dm, const bigcn_batch_t* bt, const bigcn_opts_t* o, const WFeatWs& wf,
                           const bigcn_graph_t* g, int32_t* flags, cudaStream_t st) {
  const int64_t* ei[2] = {bt->edge_index, bt->bu_edge_index};
  const int64_t E[2] = {dm->E_td, dm->E_bu};
  if (int rc = wfeat_ones(wf.ones, E[0] > E[1] ? E[0] : E[1], st)) return rc;
  for (int d = 0; d < 2; ++d) {
    if (!((o->dir_mask >> d) & 1)) continue;
    WGraph G = wf.G[d];
    G.g = g[d];
    const float* ew = dir_edge_weight(bt, d);
    if (int rc = wfeat_prep(G, ei[d], E[d], ew ? ew : wf.ones, dm->N, o->deg_by, wf.in_w[d], wf.out_w[d], flags, st))
      return rc;
  }
  return 0;
}

int batch_prepare_join(cudaStream_t st);

// active directions: order TD (0), BU (1); feat base: BU -> 0, TD -> 128 (cat order of :128)
struct Dirs {
  int n;
  int id[2];
};
static Dirs active_dirs(int mask) {
  Dirs r{0, {0, 0}};
  if (mask & BIGCN_DIR_TD) r.id[r.n++] = 0;
  if (mask & BIGCN_DIR_BU) r.id[r.n++] = 1;
  return r;
}
static const float* dir_w1(const bigcn_params_t* p, int d) { return d == 0 ? p->td_w1 : p->bu_w1; }
static const float* dir_b1(const bigcn_params_t* p, int d) { return d == 0 ? p->td_b1 : p->bu_b1; }
static const float* dir_w2(const bigcn_params_t* p, int d) { return d == 0 ? p->td_w2 : p->bu_w2; }
static const float* dir_b2(const bigcn_params_t* p, int d) { return d == 0 ? p->td_b2 : p->bu_b2; }
static float* gdir_w1(const bigcn_params_t* p, int d) { return d == 0 ? p->td_w1 : p->bu_w1; }
static float* gdir_b1(const bigcn_params_t* p, int d) { return d == 0 ? p->td_b1 : p->bu_b1; }
static float* gdir_w2(const bigcn_params_t* p, int d) { return d == 0 ? p->td_w2 : p->bu_w2; }
static float* gdir_b2(const bigcn_params_t* p, int d) { return d == 0 ? p->td_b2 : p->bu_b2; }
static int feat_base(int d) { return d == 0 ? 2 * H : 0; }

static int check_common(const bigcn_dims_t* dm, const bigcn_opts_t* o, const char* who) {
  BIGCN_CHECK_ARG(dm && o, "%s: NULL dims/opts", who);
  BIGCN_CHECK_ARG(dm->N >= 0 && dm->B >= 0 && dm->K > 0, "%s: bad dims", who);
  BIGCN_CHECK_ARG(dm->N < (1ll << 31) - 1 && dm->E_td < (1ll << 31) - 1 && dm->E_bu < (1ll << 31) - 1,
                  "%s: N/E exceed int32", who);
  BIGCN_CHECK_ARG((o->dir_mask & 3) != 0, "%s: dir_mask selects no direction", who);
  BIGCN_CHECK_ARG(o->p_drop >= 0.f && o->p_drop < 1.f, "%s: p_drop must be in [0,1)", who);
  return 0;
}
// BIGCN_GEMM_BF16: x is a dense bf16 matrix the TMA can address (16 B rows, 16 B aligned)
static int check_bf16_x(const bigcn_dims_t* dm, const bigcn_batch_t* bt, const bigcn_opts_t* o, const char* who) {
  if (o->gemm_mode != BIGCN_GEMM_BF16 || dm->N == 0) return 0;
  BIGCN_CHECK_ARG(bt->x != nullptr, "%s: gemm_mode BF16 needs a dense bf16 x (CSR input takes gemm_mode SPARSE)", who);
  BIGCN_CHECK_ARG(dm->K % 8 == 0, "%s: gemm_mode BF16 needs in_feats a multiple of 8 (16 B rows for TMA), got %lld", who,
                  (long long)dm->K);
  BIGCN_CHECK_ARG((reinterpret_cast<uintptr_t>(bt->x) & 15) == 0, "%s: gemm_mode BF16 needs x 16-byte aligned", who);
  return 0;
}

int features_forward(const bigcn_dims_t* dm, const bigcn_batch_t* bt, const bigcn_params_t* pr,
                     const bigcn_opts_t* o, float* feat, int32_t* flags, void* ws, size_t ws_bytes,
                     cudaStream_t st) {
  if (int rc = check_common(dm, o, "features_forward")) return rc;
  if (int rc = check_bf16_x(dm, bt, o, "features_forward")) return rc;
  FeatWs w = carve_features(dm, ws, ws_bytes, bt->prepared);
  const bool weighted = batch_weighted(bt);
  const WFeatWs wf = weighted ? step_wfeat(dm, bt, ws, w.total, o->edge_grad != 0) : WFeatWs{};
  BIGCN_CHECK_ARG(ws != nullptr && ws_bytes >= w.total + wf.total, "features_forward: workspace too small (%zu < %zu)",
                  ws_bytes, w.total + wf.total);
  const bool prepared = bt->prepared != nullptr;   // graph structure, root columns, CSR / CSC of x: already there
  const int64_t N = dm->N, B = dm->B, K = dm->K;
  const Dirs dirs = active_dirs(o->dir_mask);
  const bool scan_mode = o->gemm_mode == BIGCN_GEMM_FP32 || o->gemm_mode == BIGCN_GEMM_MIXED ||
                         o->gemm_mode == BIGCN_GEMM_SPARSE;
  const bool sparse = o->gemm_mode == BIGCN_GEMM_SPARSE;
  const bool dropping = o->training && o->p_drop > 0.f;
  const bool csr_in = bt->x == nullptr && N > 0;
  const int x_bf16 = o->gemm_mode == BIGCN_GEMM_BF16;
  BIGCN_CHECK_ARG(!csr_in || (sparse && bt->x_ptr && bt->x_col && bt->x_val),
                  "features_forward: x == NULL needs gemm_mode SPARSE and x_ptr / x_col / x_val");
  if (csr_in) {
    w.xs.ptr = const_cast<int32_t*>(bt->x_ptr);
    w.xs.col = const_cast<int32_t*>(bt->x_col);
    w.xs.val = const_cast<float*>(bt->x_val);
  }
  // 1. side stream (beside the X stream): structure of both directions and node_ptr -- depends on the
  //    inputs only, so it forks before anything else is queued
  SideCtx* sc = side_ctx();
  cudaStream_t ss = sc ? sc->s.side : st;
  cudaStream_t s2 = sc ? sc->side2 : st;
  if (sc && !prepared) stream_after(sc, 0, st, ss);
  if (!prepared) {
    const int64_t* ei[2] = {bt->edge_index, bt->bu_edge_index};
    const int64_t E[2] = {dm->E_td, dm->E_bu};
    int32_t* const eids[4] = {wf.G[0].in_eid, wf.G[0].out_eid, wf.G[1].in_eid, wf.G[1].out_eid};
    if (int rc = graph_prep_impl(2, ei, E, N, bt->batch, B, o->deg_by, w.g, w.node_ptr, flags, w.prep_ws,
                                 w.prep_bytes, ss, weighted ? eids : nullptr))
      return rc;
    if (weighted)
      if (int rc = wfeat_prep_dirs(dm, bt, o, wf, w.g, flags, ss)) return rc;
  }
  // 2. weights in the layouts the kernels stream
  const int n_out = dirs.n == 2 ? 128 : 64;
  {
    TransposeJobs js{};
    for (int q = 0; q < dirs.n; ++q) {
      const int d = dirs.id[q];
      if (scan_mode) js.job[js.n++] = TransposeJob{dir_w1(pr, d), K, 0, K, w.w1T, n_out, q * H};
      js.job[js.n++] = TransposeJob{dir_w2(pr, d), H + K, 0, H, w.w2aT[d], H, 0};
      js.job[js.n++] = TransposeJob{dir_w2(pr, d), H + K, H, K, w.w2bT[d], H, 0};
    }
    if (int rc = transpose_jobs_launch(js, st)) return rc;
  }
  //    second side stream: the root rows' positive columns and, without dropout, the per-tree root
  //    projection (needs the transposed W2b) -- a short chain of its own, not behind the graph prep
  if (sc) stream_after(sc, 6, st, s2);
  // training on DENSE root features (opts.dense_roots; PHEME): the root half of conv2.lin as a tiled product into z, beside
  // the X * W product; the mix kernel then adds it instead of walking K-long column lists per node
  const bool dense_roots = dropping && o->dense_roots != 0 && bt->x != nullptr && N > 0;
  const int root_splits = dense_roots ? (debug_knob(15) == 1 ? 1 : root_dense_splits(N, K)) : 0;   // knob 15 = 1: one split (tests)
  if (dense_roots) {
    RootDenseArgs a{};
    a.x = bt->x; a.rootindex = bt->rootindex; a.batch = bt->batch;
    a.N = N; a.B = B; a.K = K; a.node_id_base = bt->node_id_base;
    a.ksplit = root_splits;
    a.x_bf16 = x_bf16;
    for (int q = 0; q < dirs.n; ++q) {
      const int d = dirs.id[q];   // one split: straight into z (the mix kernel reads a node's R before it writes the node's z)
      a.w2bT[q] = w.w2bT[d]; a.r[q] = root_splits > 1 ? w.rootR[d] : w.z[d]; a.drop[q] = make_drop(o, d);
    }
    if (int rc = root_dense_forward(a, dirs.n, s2)) return rc;
  }
  {
    RootNzArgs a{bt->x, bt->rootindex, N, B, K, w.rnz_cnt, w.rnz_col, w.rnz_val, flags,
                 w.slot, w.overflow, DW2B_CAP, x_bf16};
    if (prepared) {
      // done by bigcn_batch_prepare
    } else if (csr_in) {
      if (int rc = root_nz_csr_launch(a, bt->x_ptr, bt->x_col, bt->x_val, s2)) return rc;
    } else {
      if (int rc = root_nz_launch(a, s2)) return rc;
    }
    if (!dropping) {
      RootProjArgs pa{};
      pa.cnt = w.rnz_cnt; pa.col = w.rnz_col; pa.val = w.rnz_val; pa.B = B; pa.K = K;
      for (int q = 0; q < dirs.n; ++q) {
        pa.w2bT[q] = w.w2bT[dirs.id[q]];
        pa.P[q] = w.P[dirs.id[q]];
      }
      if (int rc = root_proj_launch(pa, dirs.n, s2)) return rc;
    }
  }
  // 3. X W1^T for all active directions in one pass over X (main stream)
  if (csr_in) {
    if (int rc = xw_csr(w.xs, w.w1T, n_out, w.xw, n_out, st)) return rc;
  } else if (prepared && sparse) {   // the capture pass ran a step ahead: same entries in the same order as the fused scan
    if (int rc = xw_ell(w.xs, bt->x, w.w1T, n_out, w.xw, n_out, st)) return rc;
  } else if (sparse && !o->skip_wgrad_prep) {
    if (int rc = xw_fp32_capture(bt->x, N, K, w.w1T, n_out, w.xw, n_out, w.xs, st)) return rc;
  } else if (scan_mode) {
    if (int rc = xw_fp32(bt->x, N, K, w.w1T, n_out, w.xw, n_out, st)) return rc;
  } else {
    const float* ws[2] = {dir_w1(pr, dirs.id[0]), dirs.n == 2 ? dir_w1(pr, dirs.id[1]) : nullptr};
    if (int rc = xw_tc_weights(bt->x, N, K, ws, K, n_out, w.w1T, w.xw, n_out, o->gemm_mode, st, w.xw_part)) return rc;
  }
  // 4. the structure is needed from here on; the side stream goes on to sort the captured
  //    non-zeros of X by column for the weight gradient while the rest of the forward runs
  if (sc) {
    if (!prepared) stream_after(sc, 1, ss, st);
    stream_after(sc, 7, s2, st);
  }
  bool side_busy = false;
  if (sparse && prepared && N > 0 && !o->skip_wgrad_prep) {   // the CSR came prepared; sort it by column beside the rest of this step
    if (sc) stream_after(sc, 2, st, sc->low);
    w.xs.flags = flags;
    if (csr_in) {
      if (int rc = xs_sort_csc(w.xs, sc ? sc->low : st)) return rc;
    } else {
      if (int rc = xs_build_csc(w.xs, bt->x, true, sc ? sc->low : st)) return rc;
    }
    side_busy = sc != nullptr;
  }
  if (sparse && !prepared) {
    if (o->skip_wgrad_prep || N == 0) {
      cudaMemsetAsync(w.xs.state, 0, 4 * sizeof(int32_t), st);
    } else {
      if (sc) stream_after(sc, 2, st, sc->low);
      w.xs.flags = flags;
      if (int rc = xs_build_csc(w.xs, bt->x, !csr_in, sc ? sc->low : st)) return rc;
      side_busy = sc != nullptr;
    }
  }
  // edge-weighted batch: the sweeps read the normalised weight of every entry, and dis stands for the self-loop weights
  EntryW ew_in{};
  for (int q = 0; q < dirs.n; ++q) ew_in.w[q] = wf.in_w[dirs.id[q]];
  const float* self_w[2] = {weighted ? wf.G[0].norm_self : w.g[0].dis, weighted ? wf.G[1].norm_self : w.g[1].dis};
  // 5. conv1 propagate + relu/dropout + conv2 lin
  {
    MixArgs a{};
    a.N = N; a.K = K; a.ldxw = n_out; a.node_id_base = bt->node_id_base; a.batch = bt->batch;
    a.rnz_cnt = w.rnz_cnt; a.rnz_col = w.rnz_col; a.rnz_val = w.rnz_val;
    for (int q = 0; q < dirs.n; ++q) {
      const int d = dirs.id[q];
      MixDir& m = a.d[q];
      m.ptr = w.g[d].in_ptr; m.idx = w.g[d].in_idx; m.dis = self_w[d];
      m.lng = w.g[d].in_long; m.E = d == 0 ? dm->E_td : dm->E_bu;
      m.xw = w.xw + q * H; m.b1 = dir_b1(pr, d);
      m.w2aT = w.w2aT[d]; m.w2bT = w.w2bT[d]; m.P = w.P[d];
      m.h1 = w.h1[d]; m.a1 = w.a1[d]; m.z = w.z[d];
      m.drop = make_drop(o, d);
      m.keep = dense_roots ? nullptr : w.keep[d];
    }
    a.root_splits = root_splits;
    for (int q = 0; q < dirs.n; ++q) a.root_r[q] = root_splits > 1 ? w.rootR[dirs.id[q]] : w.z[dirs.id[q]];
    if (int rc = prop1_mix_launch(a, dirs.n, st, weighted ? &ew_in : nullptr)) return rc;
  }
  // 6. conv2 propagate + bias + relu
  {
    PropArgs a{};
    a.N = N; a.relu = 1;
    for (int q = 0; q < dirs.n; ++q) {
      const int d = dirs.id[q];
      a.d[q] = PropDir{w.g[d].in_ptr, w.g[d].in_idx, self_w[d], w.z[d], dir_b2(pr, d), w.h2[d], H, H,
                       w.g[d].in_long, d == 0 ? dm->E_td : dm->E_bu};
    }
    if (int rc = propagate_launch(a, dirs.n, st, weighted ? &ew_in : nullptr)) return rc;
  }
  // 7. readout
  {
    if (dirs.n < 2) cudaMemsetAsync(feat, 0, (size_t)B * 4 * H * sizeof(float), st);
    ReadoutArgs a{};
    a.ndir = dirs.n; a.node_ptr = w.node_ptr; a.rootindex = bt->rootindex; a.feat = feat; a.ldfeat = 4 * H;
    a.N = N; a.B = B; a.flags = flags; a.scratch = w.ro_part;
    for (int q = 0; q < dirs.n; ++q) {
      const int d = dirs.id[q];
      a.h2[q] = w.h2[d]; a.h1[q] = w.h1[d]; a.pos[q] = w.pos[d]; a.feat_base[q] = feat_base(d);
    }
    // fused_tail: the second readout pass runs inside bigcn_train_tail, in one launch with the head and gscale
    if (int rc = readout_launch(a, st, !o->fused_tail)) return rc;
  }
  // the column sort keeps running on the low-priority stream: features_backward waits for it
  // right before the sweep that needs it (event 3)
  if (side_busy) cudaEventRecord(sc->ev[3], sc->low);
  return 0;
}

// ---- the weight-independent half of a step, for a batch the caller will step on NEXT ------------------------
// graph structure of both directions + node_ptr, the root rows' positive columns, and (SPARSE) the non-zeros of
// x as CSR (its column sort follows in the consuming step): none of it depends on the parameters, so it runs on two lowest-priority streams
// beside the whole current step -- the HBM-bound pass over the next batch's x hides under the latency-bound
// kernels of this one (what the reference's DataLoader workers do for collate, BiGCN_Twitter.py:168).
int batch_prepare(const bigcn_dims_t* dm, const bigcn_batch_t* bt, const bigcn_opts_t* o, int32_t* flags, void* prepared,
                  size_t prepared_bytes, cudaStream_t st) {
  if (int rc = check_common(dm, o, "batch_prepare")) return rc;
  if (int rc = check_bf16_x(dm, bt, o, "batch_prepare")) return rc;
  PrepWs w = carve_prepared(dm, prepared, prepared_bytes);
  const bool weighted = batch_weighted(bt);
  const WFeatWs wf = weighted ? carve_prepared_wfeat(dm, prepared) : WFeatWs{};
  BIGCN_CHECK_ARG(prepared != nullptr && prepared_bytes >= w.total + wf.total,
                  "batch_prepare: buffer too small (%zu < %zu%s)", prepared_bytes, w.total + wf.total,
                  weighted ? ": bigcn_batch_prepare_edge_bytes" : "");
  const int64_t N = dm->N, B = dm->B, K = dm->K;
  const bool sparse = o->gemm_mode == BIGCN_GEMM_SPARSE;
  const bool csr_in = bt->x == nullptr && N > 0;
  BIGCN_CHECK_ARG(!csr_in || (sparse && bt->x_ptr && bt->x_col && bt->x_val),
                  "batch_prepare: x == NULL needs gemm_mode SPARSE and x_ptr / x_col / x_val");
  SideCtx* sc = side_ctx();
  cudaStream_t pa = sc ? sc->prep[0] : st, pb = sc ? sc->prep[1] : st;
  if (sc) {
    cudaEventRecord(sc->ev[8], st);
    cudaStreamWaitEvent(pa, sc->ev[8], 0);
    cudaStreamWaitEvent(pb, sc->ev[8], 0);
  }
  // stream A: x -> CSR -> CSC (the long one: one pass over x, then the column sort)
  if (sparse) {
    if (csr_in) {
      w.xs.ptr = const_cast<int32_t*>(bt->x_ptr);
      w.xs.col = const_cast<int32_t*>(bt->x_col);
      w.xs.val = const_cast<float*>(bt->x_val);
    }
    if (N == 0) {
      cudaMemsetAsync(w.xs.state, 0, 4 * sizeof(int32_t), pa);
    } else {
      // dense x: the capture only -- the next forward's product walks the ELL slots directly, and the compaction into
      // CSR and the column sort run in the consuming step, on its low-priority stream under the forward / backward
      // (awaited right before the dW1 sweep).  A caller's CSR: the sort keys now, the sort itself in the step.
      w.xs.flags = flags;
      if (!csr_in) {
        if (int rc = x_capture(bt->x, N, K, w.xs, pa)) return rc;
      } else {
        if (int rc = xs_build_csr(w.xs, bt->x, false, pa)) return rc;
      }
    }
  }
  // stream B: structure of both directions (an edge-weighted batch: with the edge ids, then its normalisation), then
  // the root columns
  {
    const int64_t* ei[2] = {bt->edge_index, bt->bu_edge_index};
    const int64_t E[2] = {dm->E_td, dm->E_bu};
    int32_t* const eids[4] = {wf.G[0].in_eid, wf.G[0].out_eid, wf.G[1].in_eid, wf.G[1].out_eid};
    if (int rc = graph_prep_impl(2, ei, E, N, bt->batch, B, o->deg_by, w.g, w.node_ptr, flags, w.prep_ws, w.prep_bytes, pb,
                                 weighted ? eids : nullptr))
      return rc;
    if (weighted)
      if (int rc = wfeat_prep_dirs(dm, bt, o, wf, w.g, flags, pb)) return rc;
    RootNzArgs a{bt->x, bt->rootindex, N, B, K, w.rnz_cnt, w.rnz_col, w.rnz_val, flags, w.slot, w.overflow, DW2B_CAP,
                 o->gemm_mode == BIGCN_GEMM_BF16};
    if (csr_in) {
      if (int rc = root_nz_csr_launch(a, bt->x_ptr, bt->x_col, bt->x_val, pb)) return rc;
    } else {
      if (int rc = root_nz_launch(a, pb)) return rc;
    }
  }
  return 0;
}
// `st` waits for everything bigcn_batch_prepare has queued so far
int batch_prepare_join(cudaStream_t st) {
  SideCtx* sc = side_ctx();
  if (!sc) return 0;
  cudaEventRecord(sc->ev[9], sc->prep[0]);
  cudaStreamWaitEvent(st, sc->ev[9], 0);
  cudaEventRecord(sc->ev[10], sc->prep[1]);
  cudaStreamWaitEvent(st, sc->ev[10], 0);
  return 0;
}

int features_backward(const bigcn_dims_t* dm, const bigcn_batch_t* bt, const bigcn_params_t* pr,
                      const bigcn_opts_t* o, const float* grad_feat, const bigcn_params_t* gr,
                      void* ws, size_t ws_bytes, cudaStream_t st) {
  if (int rc = check_common(dm, o, "features_backward")) return rc;
  if (int rc = check_bf16_x(dm, bt, o, "features_backward")) return rc;
  FeatWs w = carve_features(dm, ws, ws_bytes, bt->prepared);
  const bool weighted = batch_weighted(bt);
  const bool edge_grad = weighted && o->edge_grad != 0;
  const WFeatWs wf = weighted ? step_wfeat(dm, bt, ws, w.total, edge_grad) : WFeatWs{};
  BIGCN_CHECK_ARG(ws != nullptr && ws_bytes >= w.total + wf.total, "features_backward: workspace too small");
  const int64_t N = dm->N, B = dm->B, K = dm->K;
  const Dirs dirs = active_dirs(o->dir_mask);
  const int n_out = dirs.n == 2 ? 128 : 64;
  const bool dropping = o->training && o->p_drop > 0.f;
  const size_t nh = (size_t)(N > 0 ? N : 1) * H;
  // XW and Z are dead after forward -- unless the edge gradient reads them (after G1 is formed): T2 and G1 then go
  // to buffers of their own
  float* t2[2] = {edge_grad ? wf.t2 : w.xw, (edge_grad ? wf.t2 : w.xw) + nh};
  float* g1[2] = {edge_grad ? wf.g1 : w.z[0], edge_grad ? wf.g1 + nh : w.z[1]};
  EntryW ew_out{};
  const float* self_w[2] = {weighted ? wf.G[0].norm_self : w.g[0].dis, weighted ? wf.G[1].norm_self : w.g[1].dis};
  for (int q = 0; q < dirs.n; ++q) ew_out.w[q] = wf.out_w[dirs.id[q]];
  float* t1cat = w.h2[0];                // H2 is dead once T2 exists
  // bwd_phase: 0 = everything, 1 = all but dW1, 2 = dW1 only (lets the caller all-reduce the
  // other gradients while the second X stream runs)
  const int phase = o->bwd_phase;
  ColsumArgs db2_reduce{};
  // the dW2 / db chains on the side streams are joined AFTER the dW1 product (nothing it writes is read by them: its
  // scratch is Z (G1, consumed by the propagate before it) and H1 (dead since the forward), not T2)
  const bool join_late = phase == 0;
  SideCtx* sc = side_ctx();
  cudaStream_t ss = sc ? sc->bw[0] : st;
  cudaStream_t s2 = sc ? sc->bw[1] : st;
  if (phase == 2) goto dw1_only;
  // 1. per-tree scaled gradient gs = grad_feat / n_b and db2 (from the readout's positive counts)
  {
    GScaleArgs a{};
    a.grad_feat = grad_feat; a.node_ptr = w.node_ptr; a.B = B;
    ColsumArgs c{};
    c.nchunk = B > 0 ? gs_chunks(B) : 0;
    for (int q = 0; q < dirs.n; ++q) {
      const int d = dirs.id[q];
      a.pos[q] = w.pos[d]; a.gs[q] = w.gs[d]; a.part[q] = w.cs_part[d]; a.feat_base[q] = feat_base(d);
      c.part[q] = w.cs_part[d]; c.out[q] = gdir_b2(gr, d);
    }
    if (!o->fused_tail)   // bigcn_train_tail already wrote gs and the db2 partials (same chunking, GS_TREES)
      if (int rc = gscale_launch(a, dirs.n, st)) return rc;
    db2_reduce = c;   // summed on the side stream (below)
  }
  // 2. T2 = A-hat^T G2 with G2 = [H2 > 0] * gs[batch] formed inside the gather
  {
    PropG2Args a{};
    a.N = N; a.batch = bt->batch;
    for (int q = 0; q < dirs.n; ++q) {
      const int d = dirs.id[q];
      a.d[q] = PropG2Dir{w.g[d].out_ptr, w.g[d].out_idx, self_w[d], w.h2[d], w.gs[d], t2[d],
                         w.g[d].out_long, d == 0 ? dm->E_td : dm->E_bu};
    }
    if (int rc = propagate_g2_launch(a, dirs.n, st, weighted ? &ew_out : nullptr)) return rc;
  }
  // 3./4. on the two side streams, beside the G1 -> T1 -> dW1 chain: db2 and dW2a = T2^T A1 on one,
  //       dW2b on the other (both read T2 only)
  if (sc) {
    stream_after(sc, 0, st, ss);
    cudaStreamWaitEvent(s2, sc->ev[0], 0);
  }
  if (int rc = colsum_reduce_launch(db2_reduce, dirs.n, ss)) return rc;
  {
    OuterArgs a{};
    OuterReduceArgs r{};
    a.N = N; r.ld = H + K; r.nchunk = N > 0 ? op_chunks(N) : 0;
    for (int q = 0; q < dirs.n; ++q) {
      const int d = dirs.id[q];
      a.u[q] = t2[d]; a.v[q] = w.a1[d]; a.part[q] = w.op_part[d];
      r.part[q] = w.op_part[d]; r.dst[q] = gdir_w2(gr, d);
    }
    if (int rc = outer64_launch(a, r, dirs.n, ss)) return rc;
  }
  {
    if (!dropping) {
      SegSumArgs sg{};
      sg.node_ptr = w.node_ptr;
      for (int q = 0; q < dirs.n; ++q) {
        sg.t[q] = t2[dirs.id[q]];
        sg.out[q] = w.dP[dirs.id[q]];
      }
      if (int rc = segsum_launch(sg, B, dirs.n, s2)) return rc;
    }
    if (dropping && o->dense_roots != 0 && bt->x != nullptr && N > 0) {   // dense roots: tiled masked product (rootdense.cu)
      Dw2bDenseArgs a{};
      a.x = bt->x; a.rootindex = bt->rootindex; a.batch = bt->batch;
      a.N = N; a.B = B; a.K = K; a.ld = H + K; a.node_id_base = bt->node_id_base;
      a.nseg = dw2b_dense_segments(N, B, K);
      a.x_bf16 = o->gemm_mode == BIGCN_GEMM_BF16;
      for (int q = 0; q < dirs.n; ++q) {
        const int d = dirs.id[q];
        a.t2[q] = t2[d]; a.part[q] = w.S[d]; a.dw2[q] = gdir_w2(gr, d); a.drop[q] = make_drop(o, d);
      }
      if (int rc = dw2b_dense_backward(a, dirs.n, s2)) return rc;
    } else {
    Dw2bArgs a{};
    a.x = bt->x; a.rootindex = bt->rootindex; a.node_ptr = w.node_ptr; a.batch = bt->batch;
    a.rnz_cnt = w.rnz_cnt; a.rnz_col = w.rnz_col; a.rnz_val = w.rnz_val; a.slot = w.slot;
    a.overflow = w.overflow;
    a.N = N; a.B = B; a.K = K; a.ld = H + K; a.node_id_base = bt->node_id_base;
    for (int q = 0; q < dirs.n; ++q) {
      const int d = dirs.id[q];
      a.d[q] = Dw2bDir{t2[d], w.dP[d], gdir_w2(gr, d), w.S[d], make_drop(o, d), w.keep[d]};
    }
    if (int rc = dw2b_launch(a, dirs.n, dropping, s2)) return rc;
    }
  }
  // 5. G1 = (T2 W2a) * mask * [H1 > 0]; db1
  {
    BwdMixArgs a{};
    a.N = N; a.ldw2 = H + K; a.node_id_base = bt->node_id_base;
    ColsumArgs c{};
    c.nchunk = N > 0 ? bm_chunks(N) : 0;
    for (int q = 0; q < dirs.n; ++q) {
      const int d = dirs.id[q];
      a.d[q] = BwdMixDir{t2[d], w.a1[d], dir_w2(pr, d), g1[d], w.cs_part1[d], make_drop(o, d)};   // A1 stands in for (H1, mask)
      c.part[q] = w.cs_part1[d]; c.out[q] = gdir_b1(gr, d);
    }
    if (int rc = bwd_mix_launch(a, dirs.n, st)) return rc;
    if (sc) stream_after(sc, 2, st, ss);           // db1: ordered sum of the partials, beside T1
    if (int rc = colsum_reduce_launch(c, dirs.n, ss)) return rc;
  }
  // 5b. edge gradient: the per-edge products of both convs while XW, Z (conv2's input M), G1 and H2 are all alive
  if (edge_grad) {
    EdgeDotArgs a{};
    a.N = N; a.batch = bt->batch;
    const int64_t* ei[2] = {bt->edge_index, bt->bu_edge_index};
    for (int q = 0; q < dirs.n; ++q) {
      const int d = dirs.id[q];
      if (dir_edge_weight(bt, d) == nullptr) continue;   // no weights, no gradient: a_e stays NULL
      a.d[q] = EdgeDotDir{ei[d], d == 0 ? dm->E_td : dm->E_bu, w.xw + q * H, n_out, g1[d], w.z[d], w.h2[d], w.gs[d],
                          wf.a_e[d], wf.a_self[d]};
    }
    if (int rc = wfeat_edge_dot(a, dirs.n, st)) return rc;
    // bigcn_features_edge_grad forks from here: the rest of its chain reads a_e / a_self and the normalisation,
    // which nothing after this point overwrites
    if (sc) cudaEventRecord(sc->ev[13], st);
  }
  // 6. T1 = A-hat^T G1, both directions side by side in one [N][n_out] matrix
  {
    PropArgs a{};
    a.N = N; a.relu = 0;
    for (int q = 0; q < dirs.n; ++q) {
      const int d = dirs.id[q];
      a.d[q] = PropDir{w.g[d].out_ptr, w.g[d].out_idx, self_w[d], g1[d], nullptr, t1cat + q * H, H, n_out,
                       w.g[d].out_long, d == 0 ? dm->E_td : dm->E_bu};
    }
    if (int rc = propagate_launch(a, dirs.n, st, weighted ? &ew_out : nullptr)) return rc;
  }
  // bwd_phase 1 (the caller reduces these gradients while dW1 runs): everything but dW1 is complete at return
  if (sc && !join_late) {
    stream_after(sc, 1, ss, st);
    stream_after(sc, 7, s2, st);
  }
  if (phase == 1) return 0;
dw1_only:
  // 7. dW1 = T1^T X: a sweep over the column-sorted non-zeros (SPARSE) or one more pass over X
  {
    float* da = gdir_w1(gr, dirs.id[0]);
    float* db = dirs.n == 2 ? gdir_w1(gr, dirs.id[1]) : nullptr;
    if (o->gemm_mode == BIGCN_GEMM_SPARSE) {
      // column-sorted X: built by this step's forward on the low-priority stream (a prepared batch brought it along)
      if (sc) cudaStreamWaitEvent(st, sc->ev[3], 0);
      if (int rc = dw_sparse(w.xs, t1cat, n_out, n_out, da, db, K, st)) return rc;
    } else if (o->gemm_mode == BIGCN_GEMM_FP32) {
      if (int rc = dw_fp32(bt->x, N, K, t1cat, n_out, n_out, w.dw_part, da, K, 0, db, K, 0, st)) return rc;
    } else {   // Z (G1, or M with an edge gradient) and H1 are dead here: they hold the TF32 hi / lo split of T1 (T2 is still
               // being read by the dW2 chains)
      if (int rc = dw_tc(bt->x, N, K, t1cat, n_out, n_out, w.z[0], w.h1[0], w.dw_part, da, K, 0, db, K, 0,
                         o->gemm_mode, st))
        return rc;
    }
    if (sc && join_late) {
      stream_after(sc, 1, ss, st);
      stream_after(sc, 7, s2, st);
    }
  }
  return 0;
}

// ---- GCNConv on its own ------------------------------------------------------------
struct ConvWs {
  bigcn_graph_t g;
  float* wT;      // [K][64]
  float* xw;      // [N][64]  (backward: T)
  float* split;   // [2][N][64] TF32 hi / lo of T (tensor-core modes)
  float* cs_part;
  float* dw_part;
  void* prep_ws; size_t prep_bytes;
  size_t total;
};
static ConvWs carve_conv(int64_t N, int64_t E, int64_t K, void* ws, size_t bytes) {
  ConvWs w{};
  Carver c(ws, bytes);
  w.g.in_ptr = c.take<int32_t>(N + 1);
  w.g.out_ptr = c.take<int32_t>(N + 1);
  w.g.in_idx = c.take<int32_t>(E > 0 ? E : 1);
  w.g.out_idx = c.take<int32_t>(E > 0 ? E : 1);
  w.g.deg = c.take<int32_t>(N > 0 ? N : 1);
  w.g.dis = c.take<float>(N > 0 ? N : 1);
  w.g.rowsum = nullptr;
  w.g.in_long = c.take<int32_t>(long_ws_ints(E));
  w.g.out_long = c.take<int32_t>(long_ws_ints(E));
  w.wT = c.take<float>((size_t)K * H * 2);
  w.xw = c.take<float>((size_t)(N > 0 ? N : 1) * H);
  w.split = c.take<float>((size_t)(N > 0 ? N : 1) * H * 2);
  w.cs_part = c.take<float>((size_t)cs_chunks(N) * H);
  w.dw_part = c.take<float>(dw_partial_floats(N, K, 64));
  w.prep_bytes = graph_prep_ws_bytes(N, E, 1);
  w.prep_ws = c.take<char>(w.prep_bytes);
  w.total = align_up(c.off, 256);
  return w;
}

// column sums of a [N][64] matrix: partials per CS chunk, then ordered reduce
__global__ void __launch_bounds__(256) k_colsum_part(const float* __restrict__ g, int64_t N,
                                                     float* __restrict__ part) {
  __shared__ float red[4][H];
  const int gq = threadIdx.x >> 6, f = threadIdx.x & 63;
  const int64_t base = (int64_t)blockIdx.x * 256;
  const int64_t end = min(N, base + 256);
  float acc = 0.f;
  for (int64_t i = base + gq; i < end; i += 4) acc += g[i * H + f];
  red[gq][f] = acc;
  __syncthreads();
  if (gq == 0) part[(int64_t)blockIdx.x * H + f] = ((red[0][f] + red[1][f]) + red[2][f]) + red[3][f];
}


int colsum64_launch(const float* g, int64_t N, float* part, float* out, cudaStream_t st) {
  const int nchunk = N > 0 ? cs_chunks(N) : 0;
  if (N > 0) {
    k_colsum_part<<<nchunk, 256, 0, st>>>(g, N, part);
    BIGCN_CHECK_LAUNCH("k_colsum_part");
  }
  ColsumArgs c{};
  c.nchunk = nchunk; c.part[0] = part; c.out[0] = out;
  return colsum_reduce_launch(c, 1, st);
}

}  // namespace bigcn

using namespace bigcn;

// Two switches for tests and measurements, read at enqueue time; not part of the documented ABI.  0 is the shipped
// value of both, and every other key is ignored.
//   key 10: 9 = the LDG form of the background capture pass over x (x_capture), anything else = the TMA-fed form.
//           bench.py times the LDG form through it (its "unpaced" capture entry); tools/stepbench.py and
//           tools/capture_check.py compare the two forms.
//   key 15: 1 = one column split of the dense-root product (rootdense.cu) at every batch size, for the tests that
//           compare a fixed summation order (tests/test_gpu_bf16.py, tests/test_gpu_parity.py).
namespace bigcn {
static int g_knob10 = 0, g_knob15 = 0;
int debug_knob(int key) { return key == 10 ? g_knob10 : key == 15 ? g_knob15 : 0; }
}  // namespace bigcn
extern "C" void bigcn_debug_set(int key, int value) {
  if (key == 10) bigcn::g_knob10 = value;
  else if (key == 15) bigcn::g_knob15 = value;
}
extern "C" const char* bigcn_last_error(void) { return g_err; }
// `stream` waits for everything the library still has in flight on its internal streams
extern "C" int bigcn_join_internal_streams(bigcn_stream_t stream) {
  SideCtx* sc = side_ctx();
  if (!sc) return 0;
  cudaEventRecord(sc->ev[1], sc->s.side);
  cudaStreamWaitEvent((cudaStream_t)stream, sc->ev[1], 0);
  cudaEventRecord(sc->ev[2], sc->low);
  cudaStreamWaitEvent((cudaStream_t)stream, sc->ev[2], 0);
  cudaEventRecord(sc->ev[6], sc->side2);
  cudaStreamWaitEvent((cudaStream_t)stream, sc->ev[6], 0);
  for (cudaStream_t s : {sc->bw[0], sc->bw[1]}) {
    cudaEventRecord(sc->ev[11], s);
    cudaStreamWaitEvent((cudaStream_t)stream, sc->ev[11], 0);
  }
  return batch_prepare_join((cudaStream_t)stream);
}
// the internal low-priority stream (cudaStream_t) or NULL: lets a caching allocator be told that
// a workspace is in use there (torch: Tensor.record_stream(ExternalStream(handle)))
extern "C" void* bigcn_internal_stream(void) {
  SideCtx* sc = side_ctx();
  return sc ? (void*)sc->low : nullptr;
}
extern "C" int bigcn_version(void) { return 109; }
extern "C" int bigcn_device_ok(void) {
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return 0;
  return major == 10 ? 1 : 0;
}

extern "C" size_t bigcn_xw_scratch_floats(int64_t K, int32_t n_w) { return (size_t)2 * H * n_w * K; }

extern "C" int bigcn_xw(const float* x, int64_t N, int64_t K, const float* w0, const float* w1, int64_t ldw,
                        float* y, int64_t ldy, int32_t gemm_mode, float* scratch, bigcn_stream_t stream) {
  if (N == 0) return 0;   // empty batch: nothing to write (x / y may be NULL)
  BIGCN_CHECK_ARG(x && w0 && y && scratch, "xw: NULL argument");
  const float* ws[2] = {w0, w1};
  return xw_dispatch(x, N, K, ws, w1 ? 2 : 1, ldw, scratch, y, ldy, gemm_mode, (cudaStream_t)stream);
}

extern "C" int bigcn_propagate(const int32_t* ptr, const int32_t* idx, const float* dis, int64_t N, int64_t E,
                               int32_t* long_ws, const float* h, int64_t ldh, const float* bias, int32_t relu,
                               float* out, int64_t ldo, bigcn_stream_t stream) {
  BIGCN_CHECK_ARG((ldh % 4 == 0) && (ldo % 4 == 0), "propagate: row pitches must be multiples of 4 floats");
  BIGCN_CHECK_ARG(((reinterpret_cast<uintptr_t>(h) | reinterpret_cast<uintptr_t>(out)) & 15) == 0,
                  "propagate: h and out must be 16 B aligned");
  PropArgs a{};
  a.N = N; a.relu = relu;
  a.d[0] = PropDir{ptr, idx, dis, h, bias, out, ldh, ldo, long_ws, E};
  return propagate_launch(a, 1, (cudaStream_t)stream);
}

extern "C" size_t bigcn_colsum64_scratch_floats(int64_t N) { return (size_t)cs_chunks(N > 0 ? N : 1) * H; }

extern "C" int bigcn_colsum64(const float* g, int64_t N, float* out, float* scratch, bigcn_stream_t stream) {
  BIGCN_CHECK_ARG(N >= 0 && out && (N == 0 || (g && scratch)), "colsum64: bad arguments");
  return colsum64_launch(g, N, scratch, out, (cudaStream_t)stream);
}

extern "C" size_t bigcn_readout_scratch_floats(int64_t N, int64_t B) { return readout_scratch_floats(N, B, 1); }

extern "C" int bigcn_readout(const float* h2, const float* h1, const int32_t* node_ptr, const int64_t* rootindex,
                             int64_t N, int64_t B, float* feat, int64_t ldfeat, float* pos, float* scratch,
                             int32_t* flags, bigcn_stream_t stream) {
  BIGCN_CHECK_ARG(node_ptr && rootindex && feat && scratch && flags && (N == 0 || (h2 && h1)), "readout: NULL argument");
  BIGCN_CHECK_ARG(ldfeat >= 2 * H, "readout: ldfeat must be >= 128");
  BIGCN_CHECK_ARG((reinterpret_cast<uintptr_t>(h2) & 15) == 0, "readout: h2 must be 16 B aligned");
  ReadoutArgs a{};
  a.ndir = 1; a.node_ptr = node_ptr; a.rootindex = rootindex; a.feat = feat; a.ldfeat = ldfeat;
  a.N = N; a.B = B; a.flags = flags; a.scratch = scratch;
  a.h2[0] = h2; a.h1[0] = h1; a.pos[0] = pos; a.feat_base[0] = 0;
  return readout_launch(a, (cudaStream_t)stream);
}

extern "C" int bigcn_readout_backward(const float* grad_feat, int64_t ldg, const int32_t* node_ptr, const int64_t* batch,
                                      int64_t N, int64_t B, float* grad_h2, bigcn_stream_t stream) {
  BIGCN_CHECK_ARG(N >= 0 && B >= 0 && ldg >= H && (ldg % 4 == 0) && (N == 0 || (grad_feat && node_ptr && batch && grad_h2)),
                  "readout_backward: bad arguments");
  BIGCN_CHECK_ARG((reinterpret_cast<uintptr_t>(grad_feat) & 15) == 0, "readout_backward: grad_feat must be 16 B aligned");
  return readout_bwd_launch(grad_feat, ldg, node_ptr, batch, N, B, grad_h2, (cudaStream_t)stream);
}

extern "C" int bigcn_dropout_mask(uint64_t seed, int32_t stream_id, int64_t node_id_base, int64_t N,
                                  int64_t n_cols, float p, uint8_t* keep, bigcn_stream_t stream) {
  BIGCN_CHECK_ARG(p >= 0.f && p < 1.f, "dropout_mask: p must be in [0,1)");
  bigcn_opts_t o{};
  o.training = 1; o.p_drop = p; o.seed = seed;
  DropSpec ds = make_drop(&o, stream_id);
  return dropout_mask_launch(ds, node_id_base, N, n_cols, keep, (cudaStream_t)stream);
}

extern "C" size_t bigcn_features_workspace_bytes(const bigcn_dims_t* dims) {
  if (!dims) return 0;
  return carve_features(dims, nullptr, 0).total;
}

extern "C" size_t bigcn_features_edge_workspace_bytes(const bigcn_dims_t* dims, int32_t edge_grad) {
  if (!dims) return 0;
  return carve_features(dims, nullptr, 0).total + carve_wfeat(dims, nullptr, edge_grad != 0).total;
}

extern "C" int bigcn_features_edge_grad(const bigcn_dims_t* dims, const bigcn_batch_t* batch, const bigcn_opts_t* opts,
                                        float* d_td_w, float* d_bu_w, void* workspace, size_t workspace_bytes,
                                        bigcn_stream_t stream) {
  if (int rc = check_common(dims, opts, "features_edge_grad")) return rc;
  BIGCN_CHECK_ARG(batch != nullptr, "features_edge_grad: NULL batch");
  BIGCN_CHECK_ARG(opts->edge_grad != 0, "features_edge_grad: needs opts.edge_grad = 1 in the forward and backward calls");
  // structure and normalisation from the prepared buffer when the batch came prepared; a_e / a_self / ddeg from the
  // workspace either way
  const FeatWs w = carve_features(dims, workspace, workspace_bytes, batch->prepared);
  const WFeatWs wf = step_wfeat(dims, batch, workspace, w.total, true);
  BIGCN_CHECK_ARG(workspace != nullptr && workspace_bytes >= w.total + wf.total,
                  "features_edge_grad: workspace too small (bigcn_features_edge_workspace_bytes(dims, 1))");
  float* out[2] = {d_td_w, d_bu_w};
  const int64_t* ei[2] = {batch->edge_index, batch->bu_edge_index};
  const int64_t E[2] = {dims->E_td, dims->E_bu};
  WGradArgs a{};
  a.N = dims->N;
  a.deg_by_source = opts->deg_by == BIGCN_DEG_BY_SOURCE;
  for (int d = 0; d < 2; ++d) {
    if (out[d] == nullptr) continue;
    BIGCN_CHECK_ARG(dir_edge_weight(batch, d) != nullptr && ((opts->dir_mask >> d) & 1),
                    "features_edge_grad: the %s gradient needs that direction active and its weights in the batch",
                    d == 0 ? "TD" : "BU");
    WGraph G = wf.G[d];
    G.g = w.g[d];
    a.d[d] = WGradDir{G, ei[d], E[d], dir_edge_weight(batch, d), wf.a_e[d], wf.a_self[d], wf.ddeg[d], out[d]};
  }
  // on the low-priority stream from the event features_backward recorded after the per-edge products: the chain runs
  // underneath the backward's T1 propagate and dW1 instead of behind them, and joins the caller's stream again here
  cudaStream_t st = (cudaStream_t)stream;
  SideCtx* sc = side_ctx();
  cudaStream_t es = st;
  if (sc) {
    cudaStreamWaitEvent(sc->low, sc->ev[13], 0);
    es = sc->low;
  }
  if (int rc = wfeat_edge_grad(a, 2, es)) return rc;
  if (sc) stream_after(sc, 14, es, st);
  return 0;
}

extern "C" size_t bigcn_batch_prepare_bytes(const bigcn_dims_t* dims) {
  if (!dims) return 0;
  return carve_prepared(dims, nullptr, 0).total;
}
extern "C" size_t bigcn_batch_prepare_edge_bytes(const bigcn_dims_t* dims) {
  if (!dims) return 0;
  return carve_prepared(dims, nullptr, 0).total + carve_prepared_wfeat(dims, nullptr).total;
}
extern "C" int bigcn_batch_prepare(const bigcn_dims_t* dims, const bigcn_batch_t* batch, const bigcn_opts_t* opts,
                                   int32_t* flags, void* prepared, size_t prepared_bytes, bigcn_stream_t stream) {
  BIGCN_CHECK_ARG(batch && flags, "batch_prepare: NULL argument");
  return batch_prepare(dims, batch, opts, flags, prepared, prepared_bytes, (cudaStream_t)stream);
}
extern "C" int bigcn_batch_prepare_join(bigcn_stream_t stream) { return batch_prepare_join((cudaStream_t)stream); }

extern "C" int bigcn_features_forward(const bigcn_dims_t* dims, const bigcn_batch_t* batch,
                                      const bigcn_params_t* params, const bigcn_opts_t* opts,
                                      float* feat, int32_t* flags, void* workspace,
                                      size_t workspace_bytes, bigcn_stream_t stream) {
  BIGCN_CHECK_ARG(batch && params && feat && flags, "features_forward: NULL argument");
  return features_forward(dims, batch, params, opts, feat, flags, workspace, workspace_bytes,
                          (cudaStream_t)stream);
}

extern "C" int bigcn_train_tail(const bigcn_dims_t* dims, const bigcn_batch_t* batch, const bigcn_opts_t* opts, float* feat,
                                const int64_t* y, int64_t B_global, const float* fc_w, const float* fc_b, float* logp,
                                float* loss, float* grad_feat, float* d_fc_w, float* d_fc_b, float* scratch,
                                size_t scratch_floats, int32_t* flags, void* workspace, size_t workspace_bytes,
                                bigcn_stream_t stream) {
  BIGCN_CHECK_ARG(dims && batch && opts && feat && flags, "train_tail: NULL argument");
  if (int rc = check_common(dims, opts, "train_tail")) return rc;
  BIGCN_CHECK_ARG(opts->fused_tail && opts->dir_mask == (BIGCN_DIR_TD | BIGCN_DIR_BU),
                  "train_tail: needs opts.fused_tail = 1 (as passed to features_forward) and both directions");
  FeatWs w = carve_features(dims, workspace, workspace_bytes, batch->prepared);
  BIGCN_CHECK_ARG(workspace != nullptr && workspace_bytes >= w.total, "train_tail: workspace too small");
  const int64_t N = dims->N, B = dims->B;
  TailArgs ta{};
  ta.ro.ndir = 2; ta.ro.node_ptr = w.node_ptr; ta.ro.rootindex = batch->rootindex; ta.ro.feat = feat; ta.ro.ldfeat = 4 * H;
  ta.ro.N = N; ta.ro.B = B; ta.ro.flags = flags; ta.ro.scratch = w.ro_part;
  ta.ro.nitems = ceil_div(N > 0 ? N : 1, RO_SLICE) + B;
  ta.gs.grad_feat = grad_feat; ta.gs.node_ptr = w.node_ptr; ta.gs.B = B;
  for (int d = 0; d < 2; ++d) {
    ta.ro.h2[d] = w.h2[d]; ta.ro.h1[d] = w.h1[d]; ta.ro.pos[d] = w.pos[d]; ta.ro.feat_base[d] = feat_base(d);
    ta.gs.pos[d] = w.pos[d]; ta.gs.gs[d] = w.gs[d]; ta.gs.part[d] = w.cs_part[d]; ta.gs.feat_base[d] = feat_base(d);
  }
  return train_tail_run(ta, feat, y, B, dims->C, B_global, fc_w, fc_b, logp, loss, grad_feat, d_fc_w, d_fc_b, scratch,
                        scratch_floats, (cudaStream_t)stream);
}

extern "C" int bigcn_features_backward(const bigcn_dims_t* dims, const bigcn_batch_t* batch,
                                       const bigcn_params_t* params, const bigcn_opts_t* opts,
                                       const float* grad_feat, const bigcn_params_t* grads,
                                       void* workspace, size_t workspace_bytes,
                                       bigcn_stream_t stream) {
  BIGCN_CHECK_ARG(batch && params && grad_feat && grads, "features_backward: NULL argument");
  return features_backward(dims, batch, params, opts, grad_feat, grads, workspace, workspace_bytes,
                           (cudaStream_t)stream);
}

// ---- gradient w.r.t. x of the feature path: dX = T1cat [W1_d0; W1_d1] (SURVEY.md appendix B) ----------------------
extern "C" size_t bigcn_x_dgrad_scratch_floats(int64_t N, int64_t K, int32_t n_w) { return dx_tc_scratch_floats(N, K, n_w); }

extern "C" int bigcn_x_dgrad(const float* t, int32_t n_w, const float* w0, const float* w1, int64_t ldw, int64_t N,
                             int64_t K, float* dx, void* dx_bf16, float* scratch, bigcn_stream_t stream) {
  const float* ws[2] = {w0, w1};
  return dx_tc(t, n_w, ws, ldw, N, K, dx, dx_bf16, scratch, (cudaStream_t)stream);
}

extern "C" int bigcn_features_x_grad(const bigcn_dims_t* dims, const bigcn_params_t* params, const bigcn_opts_t* opts,
                                     float* dx, void* dx_bf16, float* scratch, void* workspace, size_t workspace_bytes,
                                     bigcn_stream_t stream) {
  if (int rc = check_common(dims, opts, "features_x_grad")) return rc;
  BIGCN_CHECK_ARG(params != nullptr, "features_x_grad: NULL params");
  const FeatWs w = carve_features(dims, workspace, workspace_bytes);
  BIGCN_CHECK_ARG(workspace != nullptr && workspace_bytes >= w.total, "features_x_grad: workspace too small");
  const Dirs dirs = active_dirs(opts->dir_mask);
  BIGCN_CHECK_ARG(dirs.n > 0, "features_x_grad: empty dir_mask");
  // T1 of the active directions, side by side: written by bigcn_features_backward, read by nothing after it
  const float* ws[2] = {dir_w1(params, dirs.id[0]), dirs.n == 2 ? dir_w1(params, dirs.id[1]) : nullptr};
  return dx_tc(w.h2[0], dirs.n, ws, dims->K, dims->N, dims->K, dx, dx_bf16, scratch, (cudaStream_t)stream);
}

// ---- ... for a CSR x: the same gradient sampled at x's stored entries (an SDDMM) ----------------------------------
extern "C" size_t bigcn_x_dgrad_csr_scratch_floats(int64_t K, int32_t n_w) { return (size_t)(K > 0 ? K : 0) * H * n_w; }

extern "C" int bigcn_x_dgrad_csr(const int32_t* ptr, const int32_t* col, int64_t N, int64_t K, int64_t nnz,
                                 const float* t, int32_t n_w, const float* w0, const float* w1, int64_t ldw, float* dval,
                                 float* scratch, bigcn_stream_t stream) {
  BIGCN_CHECK_ARG(N >= 0 && K > 0 && nnz >= 0, "x_dgrad_csr: bad dims");
  BIGCN_CHECK_ARG((n_w == 1 && w1 == nullptr) || (n_w == 2 && w1 != nullptr), "x_dgrad_csr: n_w must be 1 (w1 NULL) or 2");
  BIGCN_CHECK_ARG(ldw >= K, "x_dgrad_csr: ldw < K");
  if (N == 0 && nnz == 0) return 0;
  // col and t are read only for entries below nnz: an empty CSR may pass NULL for them
  BIGCN_CHECK_ARG(w0 && scratch && (N == 0 || ptr) && (nnz == 0 || (dval && col && t)), "x_dgrad_csr: NULL argument");
  BIGCN_CHECK_ARG(((reinterpret_cast<uintptr_t>(t) | reinterpret_cast<uintptr_t>(scratch)) & 15) == 0,
                  "x_dgrad_csr: t and scratch must be 16 B aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int n_out = H * n_w;
  TransposeJobs js{};
  js.job[js.n++] = TransposeJob{w0, ldw, 0, K, scratch, n_out, 0};
  if (n_w == 2) js.job[js.n++] = TransposeJob{w1, ldw, 0, K, scratch, n_out, H};
  if (int rc = transpose_jobs_launch(js, st)) return rc;
  return dx_csr(ptr, col, N, K, nnz, t, scratch, n_out, dval, st);
}

extern "C" int bigcn_features_x_grad_csr(const bigcn_dims_t* dims, const bigcn_batch_t* batch, const bigcn_opts_t* opts,
                                         float* dval, int64_t nnz, void* workspace, size_t workspace_bytes,
                                         bigcn_stream_t stream) {
  if (int rc = check_common(dims, opts, "features_x_grad_csr")) return rc;
  BIGCN_CHECK_ARG(batch && batch->x == nullptr && batch->x_ptr && batch->x_col,
                  "features_x_grad_csr: needs the CSR x the forward read (x NULL, x_ptr / x_col set)");
  BIGCN_CHECK_ARG(opts->gemm_mode == BIGCN_GEMM_SPARSE, "features_x_grad_csr: a CSR x runs in gemm_mode SPARSE");
  BIGCN_CHECK_ARG(nnz >= 0 && (nnz == 0 || dval), "features_x_grad_csr: bad dval / nnz");
  const FeatWs w = carve_features(dims, workspace, workspace_bytes);
  BIGCN_CHECK_ARG(workspace != nullptr && workspace_bytes >= w.total, "features_x_grad_csr: workspace too small");
  const int n_out = active_dirs(opts->dir_mask).n == 2 ? 2 * H : H;
  // T1cat [N][n_out]: written by bigcn_features_backward.  W1^T [K][n_out] in the same direction order: written by
  // bigcn_features_forward (step 2, every gemm_mode SPARSE step), and by nothing after it
  return dx_csr(batch->x_ptr, batch->x_col, dims->N, dims->K, nnz, w.h2[0], w.w1T, n_out, dval, (cudaStream_t)stream);
}

extern "C" size_t bigcn_gcnconv_workspace_bytes(int64_t N, int64_t E, int64_t K) {
  return carve_conv(N, E, K, nullptr, 0).total;
}

extern "C" int bigcn_gcnconv_forward(const float* x, int64_t N, int64_t K, const int64_t* edge_index,
                                     int64_t E, const float* w, const float* bias, int32_t deg_by,
                                     int32_t gemm_mode, float* out, int32_t* flags, void* workspace,
                                     size_t workspace_bytes, bigcn_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  BIGCN_CHECK_ARG(N >= 0 && K > 0 && E >= 0, "gcnconv_forward: bad dims");
  ConvWs cw = carve_conv(N, E, K, workspace, workspace_bytes);
  BIGCN_CHECK_ARG(workspace && workspace_bytes >= cw.total, "gcnconv_forward: workspace too small");
  const int64_t* ei[1] = {edge_index};
  const int64_t Es[1] = {E};
  if (int rc = graph_prep_impl(1, ei, Es, N, nullptr, 0, deg_by, &cw.g, nullptr, flags, cw.prep_ws,
                               cw.prep_bytes, st))
    return rc;
  const float* ws1[1] = {w};
  if (int rc = xw_dispatch(x, N, K, ws1, 1, K, cw.wT, cw.xw, H, gemm_mode, st)) return rc;
  PropArgs a{};
  a.N = N; a.relu = 0;
  a.d[0] = PropDir{cw.g.in_ptr, cw.g.in_idx, cw.g.dis, cw.xw, bias, out, H, H, cw.g.in_long, E};
  return propagate_launch(a, 1, st);
}

extern "C" int bigcn_gcnconv_backward(const float* x, int64_t N, int64_t K, int64_t E,
                                      const float* grad_out, float* dw, float* db, int32_t gemm_mode,
                                      void* workspace, size_t workspace_bytes, bigcn_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  ConvWs cw = carve_conv(N, E, K, workspace, workspace_bytes);
  BIGCN_CHECK_ARG(workspace && workspace_bytes >= cw.total, "gcnconv_backward: workspace too small");
  // db = column sums of grad_out
  const int nchunk = N > 0 ? cs_chunks(N) : 0;
  if (N > 0) {
    k_colsum_part<<<nchunk, 256, 0, st>>>(grad_out, N, cw.cs_part);
    BIGCN_CHECK_LAUNCH("k_colsum_part");
  }
  ColsumArgs c{};
  c.nchunk = nchunk; c.part[0] = cw.cs_part; c.out[0] = db;
  if (int rc = colsum_reduce_launch(c, 1, st)) return rc;
  if (gemm_mode == BIGCN_GEMM_SPARSE) gemm_mode = BIGCN_GEMM_FP32;
  // T = A-hat^T grad_out
  PropArgs a{};
  a.N = N; a.relu = 0;
  a.d[0] = PropDir{cw.g.out_ptr, cw.g.out_idx, cw.g.dis, grad_out, nullptr, cw.xw, H, H, cw.g.out_long, E};
  if (int rc = propagate_launch(a, 1, st)) return rc;
  // dw = T^T x
  if (gemm_mode == BIGCN_GEMM_FP32) return dw_fp32(x, N, K, cw.xw, H, 64, cw.dw_part, dw, K, 0, nullptr, 0, 0, st);
  return dw_tc(x, N, K, cw.xw, H, 64, cw.split, cw.split + (size_t)(N > 0 ? N : 1) * H, cw.dw_part, dw, K, 0,
               nullptr, 0, 0, gemm_mode, st);
}

// ---- GCNConv on a CSR x: BiGCN's sparse-input conv1 kernels for one direction ------------------------------------
// The workspace the forward hands to the backward holds the structure, W^T and X W^T (then T): nothing N x K and
// nothing per non-zero.  The per-non-zero buffers (sort keys, column-sorted copy, hub-column lists; BiGCN's capacity
// N * min(K, 48)) are a scratch of each call: the forward checks the columns and the capacity with k_xs_from_csr, the
// backward runs it again (no flags) and sorts by column for the dW sweep.
struct ConvCsrWs {
  bigcn_graph_t g;
  float* wT;      // [K][64]
  float* xw;      // [N][64]  (backward: T)
  float* cs_part;
  void* prep_ws; size_t prep_bytes;
  size_t total;
};
static ConvCsrWs carve_conv_csr(int64_t N, int64_t E, int64_t K, void* ws, size_t bytes) {
  ConvCsrWs w{};
  Carver c(ws, bytes);
  w.g.in_ptr = c.take<int32_t>(N + 1);
  w.g.out_ptr = c.take<int32_t>(N + 1);
  w.g.in_idx = c.take<int32_t>(E > 0 ? E : 1);
  w.g.out_idx = c.take<int32_t>(E > 0 ? E : 1);
  w.g.deg = c.take<int32_t>(N > 0 ? N : 1);
  w.g.dis = c.take<float>(N > 0 ? N : 1);
  w.g.rowsum = nullptr;
  w.g.in_long = c.take<int32_t>(long_ws_ints(E));
  w.g.out_long = c.take<int32_t>(long_ws_ints(E));
  w.wT = c.take<float>((size_t)K * H);
  w.xw = c.take<float>((size_t)(N > 0 ? N : 1) * H);
  w.cs_part = c.take<float>((size_t)cs_chunks(N) * H);
  w.prep_bytes = graph_prep_ws_bytes(N, E, 1);
  w.prep_ws = c.take<char>(w.prep_bytes);
  w.total = align_up(c.off, 256);
  return w;
}

struct ConvCsrScratch {
  XSparse xs;
  size_t total;
};
static ConvCsrScratch carve_conv_csr_scratch(int64_t N, int64_t K, void* ws, size_t bytes) {
  ConvCsrScratch w{};
  Carver c(ws, bytes);
  w.xs = xs_carve_csr(c, N, K);
  w.total = align_up(c.off, 256);
  return w;
}

// the caller's CSR in the scratch's view, the keys / row ids / capacity state written (k_xs_from_csr)
static int conv_csr_keys(ConvCsrScratch& sc, const int32_t* ptr, const int32_t* col, const float* val, int32_t* flags,
                         cudaStream_t st) {
  sc.xs.ptr = const_cast<int32_t*>(ptr);
  sc.xs.col = const_cast<int32_t*>(col);
  sc.xs.val = const_cast<float*>(val);
  sc.xs.flags = flags;
  return xs_build_csr(sc.xs, nullptr, false, st);
}

extern "C" size_t bigcn_gcnconv_csr_workspace_bytes(int64_t N, int64_t E, int64_t K) {
  return carve_conv_csr(N, E, K, nullptr, 0).total;
}

extern "C" size_t bigcn_gcnconv_csr_scratch_bytes(int64_t N, int64_t K) {
  return carve_conv_csr_scratch(N, K, nullptr, 0).total;
}

extern "C" int bigcn_gcnconv_csr_forward(const int32_t* ptr, const int32_t* col, const float* val, int64_t N, int64_t K,
                                         const int64_t* edge_index, int64_t E, const float* w, const float* bias,
                                         int32_t deg_by, float* out, int32_t* flags, void* workspace,
                                         size_t workspace_bytes, void* scratch, size_t scratch_bytes,
                                         bigcn_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  BIGCN_CHECK_ARG(N >= 0 && K > 0 && E >= 0, "gcnconv_csr_forward: bad dims");
  BIGCN_CHECK_ARG(w && flags && (N == 0 || (ptr && out)), "gcnconv_csr_forward: NULL argument");
  ConvCsrWs cw = carve_conv_csr(N, E, K, workspace, workspace_bytes);
  BIGCN_CHECK_ARG(workspace && workspace_bytes >= cw.total, "gcnconv_csr_forward: workspace too small");
  ConvCsrScratch sc = carve_conv_csr_scratch(N, K, scratch, scratch_bytes);
  BIGCN_CHECK_ARG(scratch && scratch_bytes >= sc.total, "gcnconv_csr_forward: scratch too small");
  const int64_t* ei[1] = {edge_index};
  const int64_t Es[1] = {E};
  if (int rc = graph_prep_impl(1, ei, Es, N, nullptr, 0, deg_by, &cw.g, nullptr, flags, cw.prep_ws, cw.prep_bytes, st))
    return rc;
  if (N == 0) return 0;
  TransposeJobs js{};
  js.job[js.n++] = TransposeJob{w, K, 0, K, cw.wT, H, 0};
  if (int rc = transpose_jobs_launch(js, st)) return rc;
  if (int rc = conv_csr_keys(sc, ptr, col, val, flags, st)) return rc;   // column range, capacity
  if (int rc = xw_csr(sc.xs, cw.wT, H, cw.xw, H, st)) return rc;
  PropArgs a{};
  a.N = N; a.relu = 0;
  a.d[0] = PropDir{cw.g.in_ptr, cw.g.in_idx, cw.g.dis, cw.xw, bias, out, H, H, cw.g.in_long, E};
  return propagate_launch(a, 1, st);
}

extern "C" int bigcn_gcnconv_csr_backward(const int32_t* ptr, const int32_t* col, const float* val, int64_t N,
                                          int64_t K, int64_t E, const float* grad_out, float* dw, float* db,
                                          void* workspace, size_t workspace_bytes, void* scratch, size_t scratch_bytes,
                                          bigcn_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  BIGCN_CHECK_ARG(N >= 0 && K > 0 && E >= 0 && dw && db && (N == 0 || (ptr && grad_out)),
                  "gcnconv_csr_backward: bad arguments");
  ConvCsrWs cw = carve_conv_csr(N, E, K, workspace, workspace_bytes);
  BIGCN_CHECK_ARG(workspace && workspace_bytes >= cw.total, "gcnconv_csr_backward: workspace too small");
  ConvCsrScratch sc = carve_conv_csr_scratch(N, K, scratch, scratch_bytes);
  BIGCN_CHECK_ARG(scratch && scratch_bytes >= sc.total, "gcnconv_csr_backward: scratch too small");
  if (N == 0) {
    cudaMemsetAsync(dw, 0, (size_t)H * K * sizeof(float), st);
    cudaMemsetAsync(db, 0, H * sizeof(float), st);
    return 0;
  }
  k_colsum_part<<<cs_chunks(N), 256, 0, st>>>(grad_out, N, cw.cs_part);
  BIGCN_CHECK_LAUNCH("k_colsum_part");
  ColsumArgs c{};
  c.nchunk = cs_chunks(N); c.part[0] = cw.cs_part; c.out[0] = db;
  if (int rc = colsum_reduce_launch(c, 1, st)) return rc;
  // T = A-hat^T grad_out
  PropArgs a{};
  a.N = N; a.relu = 0;
  a.d[0] = PropDir{cw.g.out_ptr, cw.g.out_idx, cw.g.dis, grad_out, nullptr, cw.xw, H, H, cw.g.out_long, E};
  if (int rc = propagate_launch(a, 1, st)) return rc;
  // dw = T^T x: the sort keys again (the forward raised the flags), the column-sorted copy, the column sweep (NaN past
  // the capacity)
  if (int rc = conv_csr_keys(sc, ptr, col, val, nullptr, st)) return rc;
  if (int rc = xs_sort_csc(sc.xs, st)) return rc;
  return dw_sparse(sc.xs, cw.xw, H, H, dw, nullptr, K, st);
}

// ---- X * W^T with the row-sparse capture, and its weight gradient, on their own -------------
struct XsWs {
  XSparse xs;
  float* wT;
  size_t total;
};
static XsWs carve_xs(int64_t N, int64_t K, void* ws, size_t bytes) {
  XsWs w{};
  Carver c(ws, bytes);
  w.xs = xs_carve(c, N, K);
  w.wT = c.take<float>((size_t)K * 128);
  w.total = align_up(c.off, 256);
  return w;
}
extern "C" size_t bigcn_xsparse_workspace_bytes(int64_t N, int64_t K) { return carve_xs(N, K, nullptr, 0).total; }

extern "C" int bigcn_xw_sparse(const float* x, int64_t N, int64_t K, const float* w0, const float* w1, int64_t ldw,
                               float* y, int64_t ldy, int32_t build_csc, int32_t* flags, void* workspace,
                               size_t workspace_bytes, bigcn_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  BIGCN_CHECK_ARG(N >= 0 && K > 0 && w0 && flags && (N == 0 || (x && y)), "xw_sparse: bad arguments");
  XsWs w = carve_xs(N, K, workspace, workspace_bytes);
  BIGCN_CHECK_ARG(workspace && workspace_bytes >= w.total, "xw_sparse: workspace too small");
  if (N == 0) {
    cudaMemsetAsync(w.xs.state, 0, 4 * sizeof(int32_t), st);
    return 0;
  }
  const int n_w = w1 ? 2 : 1;
  TransposeJobs js{};
  js.job[js.n++] = TransposeJob{w0, ldw, 0, K, w.wT, H * n_w, 0};
  if (w1) js.job[js.n++] = TransposeJob{w1, ldw, 0, K, w.wT, H * n_w, H};
  if (int rc = transpose_jobs_launch(js, st)) return rc;
  if (int rc = xw_fp32_capture(x, N, K, w.wT, H * n_w, y, ldy, w.xs, st)) return rc;
  if (!build_csc) {
    cudaMemsetAsync(w.xs.state, 0, 4 * sizeof(int32_t), st);
    return 0;
  }
  w.xs.flags = flags;
  return xs_build_csc(w.xs, x, true, st);
}

// the pass over x of bigcn_batch_prepare on its own: capture of the non-zeros into the ELL slots of a
// bigcn_xw_sparse workspace (no product); with build_csr != 0 also the exclusive scan + compaction into CSR
extern "C" int bigcn_x_capture(const float* x, int64_t N, int64_t K, int32_t build_csr, int32_t* flags, void* workspace,
                               size_t workspace_bytes, bigcn_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  BIGCN_CHECK_ARG(N >= 0 && K > 0 && flags && (N == 0 || x), "x_capture: bad arguments");
  XsWs w = carve_xs(N, K, workspace, workspace_bytes);
  BIGCN_CHECK_ARG(workspace && workspace_bytes >= w.total, "x_capture: workspace too small");
  if (N == 0) return 0;
  if (int rc = x_capture(x, N, K, w.xs, st)) return rc;
  if (!build_csr) return 0;
  w.xs.flags = flags;
  return xs_build_csr(w.xs, x, true, st);
}

extern "C" int bigcn_xw_wgrad_sparse(int64_t N, int64_t K, const float* t, int32_t n_w, float* dw0, float* dw1,
                                     int64_t ldw, void* workspace, size_t workspace_bytes, bigcn_stream_t stream) {
  BIGCN_CHECK_ARG(t && dw0 && (n_w == 1 || (n_w == 2 && dw1)), "xw_wgrad_sparse: bad arguments");
  XsWs w = carve_xs(N, K, workspace, workspace_bytes);
  BIGCN_CHECK_ARG(workspace && workspace_bytes >= w.total, "xw_wgrad_sparse: workspace too small");
  return dw_sparse(w.xs, t, H * n_w, H * n_w, dw0, dw1, ldw, (cudaStream_t)stream);
}

// device pointers of the CSR / CSC built in a bigcn_xw_sparse workspace (tests, sparse loaders)
extern "C" int bigcn_xsparse_view(int64_t N, int64_t K, void* workspace, size_t workspace_bytes, int32_t** state,
                                  int32_t** ptr, int32_t** col, float** val, int32_t** cptr, int32_t** crow,
                                  float** cval) {
  XsWs w = carve_xs(N, K, workspace, workspace_bytes);
  BIGCN_CHECK_ARG(workspace && workspace_bytes >= w.total, "xsparse_view: workspace too small");
  *state = w.xs.state; *ptr = w.xs.ptr; *col = w.xs.col; *val = w.xs.val;
  *cptr = w.xs.cptr; *crow = w.xs.crow; *cval = w.xs.cval;
  return 0;
}

// ---- weight gradient of X * W^T on its own (the autograd transpose of GCNConv.lin) -------
extern "C" size_t bigcn_xw_wgrad_scratch_floats(int64_t N, int64_t K, int32_t n_w) {
  const int n_out = H * n_w;
  return dw_partial_floats(N, K, n_out) + (size_t)2 * (size_t)(N > 0 ? N : 1) * n_out;
}

extern "C" int bigcn_xw_wgrad(const float* x, int64_t N, int64_t K, const float* t, int32_t n_w, float* dw0,
                              float* dw1, int64_t ldw, int32_t gemm_mode, float* scratch,
                              bigcn_stream_t stream) {
  // N = 0 writes zeros; x and t may then be NULL (an empty torch tensor has no storage)
  BIGCN_CHECK_ARG((N == 0 || (x && t)) && dw0 && scratch && (n_w == 1 || (n_w == 2 && dw1)), "xw_wgrad: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const int n_out = H * n_w;
  float* partial = scratch;
  float* hi = scratch + dw_partial_floats(N, K, n_out);
  float* lo = hi + (size_t)(N > 0 ? N : 1) * n_out;
  if (gemm_mode == BIGCN_GEMM_FP32 || gemm_mode == BIGCN_GEMM_SPARSE)
    return dw_fp32(x, N, K, t, n_out, n_out, partial, dw0, ldw, 0, dw1, ldw, 0, st);
  return dw_tc(x, N, K, t, n_out, n_out, hi, lo, partial, dw0, ldw, 0, dw1, ldw, 0, gemm_mode, st);
}
