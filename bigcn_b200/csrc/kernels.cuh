// Argument structs and launchers shared between the kernel files and api.cu.
#pragma once
#include "common.cuh"

namespace bigcn {

constexpr int CS_ROWS = 256;  // rows per CTA for column-sum partials
constexpr int GS_TREES = 4;   // trees per CTA in k_gscale (= trees per CTA of the fused tail, k_train_tail)
constexpr int BM_ROWS = 128;  // rows per CTA in k_bwd_mix (8 warps x 16 rows)
constexpr int OP_ROWS = 128;  // rows per CTA in k_outer64
constexpr int DW2B_ROWS = 128; // rows per CTA in k_dw2b_part
constexpr int DW2B_CAP = 64;   // root slots per tree on the sparse-root fast path
constexpr int LONG_ROW = 32;         // CSR rows with more in-edges are split (gather.cuh)
constexpr int LONG_MAX_CHUNKS = 64;  // at most this many chunks per hub row
size_t long_ws_ints(int64_t E);

// eids (optional): {in_eid, out_eid} per direction -- the edge id behind every CSR entry (weighted.cu)
int graph_prep_impl(int32_t, const int64_t* const*, const int64_t*, int64_t, const int64_t*, int64_t,
                    int32_t, const bigcn_graph_t*, int32_t*, int32_t*, void*, size_t, cudaStream_t,
                    int32_t* const* eids = nullptr);
size_t graph_prep_ws_bytes(int64_t N, int64_t Emax, int ndir);
int xw_fp32(const float*, int64_t, int64_t, const float*, int, float*, int64_t, cudaStream_t);
int transpose_weight(const float*, int64_t, int64_t, int64_t, float*, int64_t, int64_t, cudaStream_t);
struct TransposeJob { const float* w; int64_t ldw, k0, K; float* wt; int64_t ldwt, col0; };
struct TransposeJobs { TransposeJob job[6]; int n; };
int transpose_jobs_launch(const TransposeJobs&, cudaStream_t);
size_t dw_partial_floats(int64_t N, int64_t K, int n_out);
int dw_reduce_launch(const float* partial, int nchunk, int64_t K, int n_out, float* dw_a, int64_t ldw_a,
                     int64_t k0_a, float* dw_b, int64_t ldw_b, int64_t k0_b, cudaStream_t st);
int dw_tc(const float* x, int64_t N, int64_t K, const float* t, int64_t ldt, int n_out, float* hi_scratch,
          float* lo_scratch, float* partial, float* dw_a, int64_t ldw_a, int64_t k0_a, float* dw_b, int64_t ldw_b, int64_t k0_b,
          int mode, cudaStream_t st);
int dw_fp32(const float*, int64_t, int64_t, const float*, int64_t, int, float*, float*, int64_t, int64_t,
            float*, int64_t, int64_t, cudaStream_t);
size_t dx_tc_scratch_floats(int64_t N, int64_t K, int n_w);
int dx_tc(const float* t, int n_w, const float* const* w, int64_t ldw, int64_t N, int64_t K, float* dx, void* dx_bf16,
          float* scratch, cudaStream_t st);

// gcn_norm with edge weights (weighted.cu): the structure of one direction and its normalisation
struct WGraph {
  bigcn_graph_t g;        // in/out CSR (deg / dis of the unweighted prep are scratch here)
  int32_t* in_eid;        // [E] edge id of every by-target CSR entry
  int32_t* out_eid;       // [E] edge id of every by-source CSR entry
  int32_t* loop_eid;      // [N] last self-loop edge on the node, or -1
  float* self_w;          // [N]
  float* dis;             // [N] weighted deg^-1/2
  float* norm_e;          // [E] per edge id (0 for self-loop / out-of-range edges)
  float* norm_self;       // [N]
};
// edge-weighted batch: the normalised weight of every entry of the CSR a sweep walks, per direction (weighted.cu);
// the launchers take NULL for the unweighted form
struct EntryW { const float* w[2]; };
// per direction of an edge-weighted feature path (weighted.cu): gcn_norm with weights on top of the feature path's
// graph prep, the normalised weights in both CSR orders, NaN / negative-degree checks (BIGCN_FLAG_EDGE_WEIGHT)
int wfeat_ones(float* ones, int64_t n, cudaStream_t st);
int wfeat_prep(const WGraph& G, const int64_t* ei, int64_t E, const float* w, int64_t N, int32_t deg_by, float* in_w,
               float* out_w, int32_t* flags, cudaStream_t st);
struct EdgeDotDir { const int64_t* ei; int64_t E; const float* xw; int64_t ldxw; const float* g1; const float* m;
                    const float* h2; const float* gs; float* a_e; float* a_self; };
struct EdgeDotArgs { EdgeDotDir d[2]; int64_t N; const int64_t* batch; };
int wfeat_edge_dot(const EdgeDotArgs& a, int ndir, cudaStream_t st);
// the chain from dL/dnorm through the normalisation to dL/dw, per direction (dw == NULL: direction skipped); both
// directions in one launch per kernel (k_w_ddeg, k_w_dweight; the direction index in grid.y)
struct WGradDir { WGraph G; const int64_t* ei; int64_t E; const float* w; const float* a_e; const float* a_self;
                  float* ddeg; float* dw; };
struct WGradArgs { WGradDir d[2]; int64_t N; int32_t deg_by_source; };
int wfeat_edge_grad(const WGradArgs& a, int ndir, cudaStream_t st);
struct PropDir { const int32_t* ptr; const int32_t* idx; const float* dis; const float* h; const float* bias; float* out; int64_t ldh, ldo; int32_t* lng; int64_t E; };
struct PropArgs { PropDir d[2]; int64_t N; int32_t relu; int32_t cb; };
int propagate_launch(const PropArgs&, int, cudaStream_t, const EntryW* ew = nullptr);
struct RootNzArgs { const float* x; const int64_t* rootindex; int64_t N, B, K; int32_t* cnt; int32_t* col; float* val; int32_t* flags; int32_t* slot; int32_t* overflow; int32_t cap;
                    int32_t x_bf16;   /* x holds bf16 (BIGCN_GEMM_BF16) */ };
int root_nz_launch(const RootNzArgs&, cudaStream_t);
int root_nz_csr_launch(const RootNzArgs&, const int32_t*, const int32_t*, const float*, cudaStream_t);
struct RootProjArgs { const int32_t* cnt; const int32_t* col; const float* val; const float* w2bT[2]; float* P[2]; int64_t B, K; };
int root_proj_launch(const RootProjArgs&, int, cudaStream_t);
struct MixDir { const int32_t* ptr; const int32_t* idx; const float* dis; const float* xw; const float* b1; const float* w2aT; const float* w2bT; const float* P; float* h1; float* a1; float* z; DropSpec drop; int32_t* lng; int64_t E; unsigned long long* keep; };
struct MixArgs { MixDir d[2]; int64_t N, K, ldxw; int32_t cb; int64_t node_id_base; const int64_t* batch; const int32_t* rnz_cnt; const int32_t* rnz_col; const float* rnz_val;
                 int32_t root_splits;    /* training, dense roots (rootdense.cu): > 0 = the root half comes as this many
                                            partial sums root_r[d] + s * N * 64, added in order; the list walk is skipped */
                 const float* root_r[2]; };
int prop1_mix_launch(const MixArgs&, int, cudaStream_t, const EntryW* ew = nullptr);
// tcgen05 form (mix_tc.cu): sweep + activate, then the 64 x 64 product on the tensor cores with the root part in the epilogue
bool mix_tc_available();
size_t mix_tc_scratch_floats();
int mix_tc_split_weights(const float* const* w2, int ndir, int64_t ldw2, float* scratch, cudaStream_t);
int mix_tc_forward(const MixArgs&, int ndir, float* scratch, cudaStream_t);
constexpr int RO_SLICE = 512;  // rows per readout slice
struct ReadoutArgs { const float* h2[2]; const float* h1[2]; float* pos[2]; int feat_base[2]; int ndir; const int32_t* node_ptr; const int64_t* rootindex; float* feat; int64_t ldfeat; int64_t N, B; int32_t* flags; float* scratch; int64_t nitems; };
int readout_launch(const ReadoutArgs&, cudaStream_t, bool with_final = true);
#ifdef __CUDACC__
// One tree's readout, second pass (thread = column f of tree b): the slice partials in slice order, the divide,
// the positive counts the backward uses for db2, and the root row of H1; writes feat / pos and hands the values back
// (k_readout_final, and the fused tail k_train_tail which goes on with the head in the same launch).
__device__ __forceinline__ void readout_final_tree(const ReadoutArgs& a, int64_t b, int f, float (&mean)[2], float (&root)[2],
                                                   float (&cnt_out)[2]) {
  const int s = a.node_ptr[b], e = a.node_ptr[b + 1];
  const int n = e - s;
  int64_t r = -1;
  if (n > 0) {
    r = a.rootindex[b];
    if (r < 0 || r >= a.N) {
      if (f == 0) atomicOr(a.flags, BIGCN_FLAG_ROOT_RANGE);
      r = -1;
    }
  }
  for (int d = 0; d < a.ndir; ++d) {
    float sum = 0.f, cnt = 0.f;
    if (n > 0) {
      const int64_t x0 = s / RO_SLICE + b, x1 = (e - 1) / RO_SLICE + b;
      for (int64_t x = x0; x <= x1; ++x) {
        const float* p = a.scratch + (((int64_t)d * a.nitems + x) * 2) * H + f;
        sum += p[0];
        cnt += p[H];
      }
    }
    if (a.pos[d]) a.pos[d][b * H + f] = cnt;
    float* fr = a.feat + b * a.ldfeat + a.feat_base[d];
    mean[d] = __fdiv_rn(sum, (float)(n > 0 ? n : 1));
    root[d] = r >= 0 ? a.h1[d][r * H + f] : 0.f;
    cnt_out[d] = cnt;
    fr[f] = mean[d];
    fr[H + f] = root[d];
  }
}
#endif
size_t readout_scratch_floats(int64_t N, int64_t B, int ndir);
int readout_bwd_launch(const float*, int64_t, const int32_t*, const int64_t*, int64_t, int64_t, float*, cudaStream_t);
struct GScaleArgs { const float* grad_feat; const float* pos[2]; float* gs[2]; float* part[2]; int feat_base[2]; const int32_t* node_ptr; int64_t B; };
int gscale_launch(const GScaleArgs&, int, cudaStream_t);
// readout-final + head (fc, log_softmax, nll gradient, grad_feat) + gscale in one launch (head.cu)
struct TailArgs { ReadoutArgs ro; GScaleArgs gs; const int64_t* y; int C; float inv_bg; const float* W; const float* bias; float* logp; float* dl; float* gfeat; float* lossvec; };
int train_tail_launch(const TailArgs&, cudaStream_t);
int train_tail_run(TailArgs ta, const float* feat, const int64_t* y, int64_t B, int64_t C, int64_t B_global, const float* fc_w,
                   const float* fc_b, float* logp, float* loss, float* grad_feat, float* d_fc_w, float* d_fc_b, float* scratch,
                   size_t scratch_floats, cudaStream_t st);
struct PropG2Dir { const int32_t* ptr; const int32_t* idx; const float* dis; const float* h2; const float* gs; float* out; int32_t* lng; int64_t E; };
struct PropG2Args { PropG2Dir d[2]; int64_t N; const int64_t* batch; int32_t cb; };
int propagate_g2_launch(const PropG2Args&, int, cudaStream_t, const EntryW* ew = nullptr);
struct ColsumArgs { const float* part[4]; float* out[4]; int nchunk; };
int colsum_reduce_launch(const ColsumArgs&, int, cudaStream_t);
struct BwdMixDir { const float* t2; const float* h1 /* A1 = dropout(relu(H1)): > 0 where kept and positive */; const float* w2; float* g1; float* part; DropSpec drop; };
struct BwdMixArgs { BwdMixDir d[2]; int64_t N, ldw2, node_id_base; };
int bwd_mix_launch(const BwdMixArgs&, int, cudaStream_t);
int mix_tc_backward(const BwdMixArgs&, int ndir, const float* scratch, cudaStream_t);
struct OuterArgs { const float* u[2]; const float* v[2]; float* part[2]; int64_t N; };
struct OuterReduceArgs { const float* part[2]; float* dst[2]; int64_t ld; int nchunk; };
int outer64_launch(const OuterArgs&, const OuterReduceArgs&, int, cudaStream_t);
struct SegSumArgs { const float* t[2]; float* out[2]; const int32_t* node_ptr; };
int segsum_launch(const SegSumArgs&, int64_t, int, cudaStream_t);
struct Dw2bDir { const float* t2; const float* dP; float* dw2; float* S; DropSpec drop; const unsigned long long* keep; };
struct Dw2bArgs { Dw2bDir d[2]; const float* x; const int64_t* rootindex; const int32_t* node_ptr; const int64_t* batch; const int32_t* rnz_cnt; const int32_t* rnz_col; const float* rnz_val; const int32_t* slot; const int32_t* overflow; int64_t N, B, K, ld, node_id_base; };
int dw2b_launch(const Dw2bArgs&, int, bool, cudaStream_t);
// dense root features in training mode (rootdense.cu): the root half of conv2.lin and its weight gradient as tiled products
struct RootDenseArgs {
  const float* x; const int64_t* rootindex; const int64_t* batch;
  int64_t N, B, K, node_id_base;
  const float* w2bT[2];   // [K][64]
  float* r[2];            // [ksplit][N][64]: sum over the split's columns of keep * relu(x_root) * W2b^T (unscaled)
  int32_t ksplit;         // column ranges summed by different CTAs (small batches: a CTA's chain of K / 32 chunks is the
                          // latency of the whole pass); the consumer adds the partials in split order
  DropSpec drop[2];
  int32_t x_bf16;         // x holds bf16 (BIGCN_GEMM_BF16)
};
constexpr int64_t RD_CAP_ROWS = 32768;   // rows of split partials per direction the workspace holds
int root_dense_splits(int64_t N, int64_t K);
struct Dw2bDenseArgs {
  const float* x; const int64_t* rootindex; const int64_t* batch;
  int64_t N, B, K, ld, node_id_base, seg_rows;
  int nseg;
  const float* t2[2];     // [N][64]
  float* part[2];         // [nseg][K][64]
  float* dw2[2];          // conv2.lin.weight gradient [64][64 + K]
  DropSpec drop[2];
  int32_t x_bf16;         // x holds bf16 (BIGCN_GEMM_BF16)
};
int root_dense_forward(const RootDenseArgs&, int ndir, cudaStream_t);
int dw2b_dense_segments(int64_t N, int64_t B, int64_t K);
int dw2b_dense_backward(const Dw2bDenseArgs&, int ndir, cudaStream_t);
int dw2b_blocks(int64_t N);
int dropout_mask_launch(const DropSpec&, int64_t, int64_t, int64_t, uint8_t*, cudaStream_t);
int cs_chunks(int64_t N);
int gs_chunks(int64_t B);
int bm_chunks(int64_t N);
int op_chunks(int64_t N);
int xw_tc_weights(const float* x, int64_t N, int64_t K, const float* const* w, int64_t ldw, int n_out,
                  float* scratch, float* y, int64_t ldy, int mode, cudaStream_t st, float* partial = nullptr);
size_t xw_tc_partial_floats();
bool xw_tc_available();

// ---- row-sparse view of X (xsparse.cu) -------------------------------------------------------
constexpr int XS_ELL = 32;           // non-zeros per row the forward scan captures in place
constexpr int XS_CAP_PER_ROW = 48;   // the CSR / CSC buffers hold N * min(K, 48) entries
struct XSparse {
  int64_t N, K, cap;
  int32_t* state;     // [0] nnz the sort / sweep work on, [1] 1 = more non-zeros than cap
  int32_t* cnt;       // [N]    non-zeros per row (exact)
  int32_t* ell_col;   // [N][XS_ELL]
  float* ell_val;     // [N][XS_ELL]
  int32_t* ptr;       // [N+1]  CSR
  int32_t* col;       // [cap]
  int32_t* row;       // [cap]
  float* val;         // [cap]
  int32_t* keys[2];   // radix ping-pong
  int32_t* perm[2];
  int32_t* hist;
  int32_t* bsum;
  int32_t* cptr;      // [K+1]  CSC
  int32_t* crow;      // [cap]
  float* cval;        // [cap]
  int32_t* clong[2];  // hub-column lists, one per 64-output half (each owns its partials / arrival counters)
  int32_t* flags;     // caller's violation word (BIGCN_FLAG_X_NOT_SPARSE)
};
int debug_knob(int key);
int64_t xs_capacity(int64_t N, int64_t K);
XSparse xs_carve(Carver& c, int64_t N, int64_t K);
// st_tail: leave the last two launches (xs_sort_finish) to the caller
int xs_build_csc(const XSparse& x, const float* x_dense, bool from_capture, cudaStream_t st, bool st_tail = false);
int xs_build_csr(const XSparse& x, const float* x_dense, bool from_capture, cudaStream_t st);
int xs_sort_csc(const XSparse& x, cudaStream_t st, bool st_tail = false);
int xs_sort_finish(const XSparse& x, cudaStream_t st);
int dw_sparse(const XSparse& x, const float* t, int64_t ldt, int n_out, float* dw_a, float* dw_b, int64_t ldw,
              cudaStream_t st);
int xw_fp32_capture(const float*, int64_t, int64_t, const float*, int, float*, int64_t, const XSparse&, cudaStream_t);
int xw_csr(const XSparse& x, const float* wt, int n_out, float* y, int64_t ldy, cudaStream_t st, bool check_state = false);
int x_capture(const float* x, int64_t N, int64_t K, const XSparse& xs, cudaStream_t st);
int xw_ell(const XSparse& xs, const float* x, const float* wt, int n_out, float* y, int64_t ldy, cudaStream_t st);
// dval[e] = t[i] . wt[col[e]] for every stored entry e = (i, col[e]) of the CSR (ptr, col); 0 for e in [ptr[N], nnz)
int dx_csr(const int32_t* ptr, const int32_t* col, int64_t N, int64_t K, int64_t nnz, const float* t, const float* wt,
           int n_out, float* dval, cudaStream_t st);

// fork / join onto the library's side stream (independent short kernels run beside the main chain)
struct SideStream {
  cudaStream_t side;
};
cudaStream_t side_fork(cudaStream_t main_st);   // the side stream, ordered after everything queued on main so far
void side_join(cudaStream_t main_st);           // main waits for everything queued on the side stream


}  // namespace bigcn
