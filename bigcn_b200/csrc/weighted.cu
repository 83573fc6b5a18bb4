// Edge-weighted GCNConv (SURVEY.md 8f N3): conv(x, edge_index, edge_weight) as the reference's
// EBGCN calls it (model/Twitter/EBGCN.py:84 `self.conv2(x, edge_index, edge_weight=edge_pred)`,
// BU twin :181), and gcn_norm with weights as explain_PHEME.py:62-63 calls it directly.
//
// Replaces, for that call: gcn_norm / add_remaining_self_loops with weights, the message
// `norm * x_j`, the sum-aggregate at the target [torch_geometric], and their autograd -- including
// the gradient that reaches the edge weights (edge_pred is produced by a trained sub-network) both
// directly and through the degree normalisation, and the gradient w.r.t. x (EBGCN feeds conv2 a
// batch-normalised tensor that depends on conv1).
//
//   self_w[i] = weight of the (last) self-loop edge on i in the list, else 1      (fill_value = 1)
//   deg[i]    = sum of w_e over the non-loop edges with target i (source i for deg_by = source),
//               added in edge-list order, then + self_w[i]                         (scatter_add, COO')
//   dis[i]    = 1 / sqrt(deg[i]), inf -> 0
//   norm_e    = (dis[row] * w_e) * dis[col],   norm_self[i] = (dis[i] * self_w[i]) * dis[i]
//   out[i]    = sum over in-edges in edge-list order of norm_e * h[row_e], then + norm_self[i] * h[i], + bias
//
// Structure: the integer graph prep of graph_prep.cu with the edge id carried as the sort payload
// (in_eid / out_eid), so both CSRs can look weights up per entry.  Every sum walks a CSR row in
// edge-list order (separate multiply and add, no atomics on floats): results are deterministic
// and the forward equals the oracle's index_add_ order bit for bit.  Warp per row: these kernels
// are the generic form (arbitrary graphs and weights), not the tuned sweep of gather.cuh.
#include "kernels.cuh"

namespace bigcn {

// ---- pass 1: which edge supplies a node's self-loop weight ----------------------------------
__global__ void k_w_loops(const int64_t* __restrict__ ei, int64_t E, int64_t N, int32_t* loop_eid) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = ei[e], c = ei[E + e];
    if (r == c && r >= 0 && r < N) atomicMax(loop_eid + r, (int32_t)e);   // "last write wins" of the CPU index_put
  }
}

// sum of w over one CSR row in order (lanes load, one running sum): every lane returns the total
__device__ __forceinline__ float row_weight_sum(const int32_t* __restrict__ eid, const float* __restrict__ w, int s,
                                                int e, int lane) {
  float acc = 0.f;
  for (int b = s; b < e; b += 32) {
    const int n = min(32, e - b);
    float p = 0.f;
    if (lane < n) p = w[eid[b + lane]];
    for (int l = 0; l < n; ++l) acc = __fadd_rn(acc, __shfl_sync(FULL_MASK, p, l));
  }
  return acc;
}

// ---- pass 2: weighted degree, dis, self weights (warp per node) ------------------------------
__global__ void __launch_bounds__(256) k_w_deg(WGraph G, const float* __restrict__ w, int64_t N, int deg_by_source) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarp = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int32_t* ptr = deg_by_source ? G.g.out_ptr : G.g.in_ptr;
  const int32_t* eid = deg_by_source ? G.out_eid : G.in_eid;
  for (int64_t i = warp0; i < N; i += nwarp) {
    float acc = row_weight_sum(eid, w, ptr[i], ptr[i + 1], lane);
    const int32_t le = G.loop_eid[i];
    const float sw = le >= 0 ? w[le] : 1.0f;
    acc = __fadd_rn(acc, sw);
    float d = __fdiv_rn(1.0f, __fsqrt_rn(acc));     // torch CPU pow(-0.5)
    if (isinf(d)) d = 0.f;                           // masked_fill(dis == inf, 0)
    if (lane == 0) {
      G.self_w[i] = sw;
      G.dis[i] = d;
      G.norm_self[i] = __fmul_rn(__fmul_rn(d, sw), d);
    }
  }
}

// ---- pass 3: norm per edge id ----------------------------------------------------------------
__global__ void k_w_norm(WGraph G, const int64_t* __restrict__ ei, const float* __restrict__ w, int64_t E, int64_t N) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = ei[e], c = ei[E + e];
    const bool valid = r != c && r >= 0 && r < N && c >= 0 && c < N;
    G.norm_e[e] = valid ? __fmul_rn(__fmul_rn(G.dis[r], w[e]), G.dis[c]) : 0.f;
  }
}

// ---- propagate: out[i] = sum_entries norm[eid] * h[idx] (+ norm_self[i] h[i]) (+ bias) -------
// warp per row, lane owns 2 of the 64 columns; (index, norm) pairs of 32 entries per coalesced load,
// rows gathered four at a time, accumulated strictly in entry order.  RELU: relu of the sum (EBGCN's conv2, ebgcn.cu).
template <bool RELU>
__global__ void __launch_bounds__(256) k_w_propagate(const int32_t* __restrict__ ptr, const int32_t* __restrict__ idx,
                                                     const int32_t* __restrict__ eid, const float* __restrict__ norm_e,
                                                     const float* __restrict__ norm_self, const float* __restrict__ h,
                                                     int64_t ldh, const float* __restrict__ bias, float* __restrict__ out,
                                                     int64_t ldo, int64_t N) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarp = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i = warp0; i < N; i += nwarp) {
    const int s = ptr[i], e = ptr[i + 1];
    float2 acc = make_float2(0.f, 0.f);
    for (int b = s; b < e; b += 32) {
      const int n = min(32, e - b);
      int src = 0;
      float nr = 0.f;
      if (lane < n) {
        src = idx[b + lane];
        nr = norm_e[eid[b + lane]];
      }
      int l = 0;
      for (; l + 4 <= n; l += 4) {
        float2 v[4];
        float wv[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int sj = __shfl_sync(FULL_MASK, src, l + q);
          wv[q] = __shfl_sync(FULL_MASK, nr, l + q);
          v[q] = *reinterpret_cast<const float2*>(h + (int64_t)sj * ldh + 2 * lane);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          acc.x = __fadd_rn(acc.x, __fmul_rn(wv[q], v[q].x));
          acc.y = __fadd_rn(acc.y, __fmul_rn(wv[q], v[q].y));
        }
      }
      for (; l < n; ++l) {
        const int sj = __shfl_sync(FULL_MASK, src, l);
        const float wq = __shfl_sync(FULL_MASK, nr, l);
        const float2 v = *reinterpret_cast<const float2*>(h + (int64_t)sj * ldh + 2 * lane);
        acc.x = __fadd_rn(acc.x, __fmul_rn(wq, v.x));
        acc.y = __fadd_rn(acc.y, __fmul_rn(wq, v.y));
      }
    }
    const float ns = norm_self[i];
    const float2 hv = *reinterpret_cast<const float2*>(h + i * ldh + 2 * lane);
    acc.x = __fadd_rn(acc.x, __fmul_rn(ns, hv.x));
    acc.y = __fadd_rn(acc.y, __fmul_rn(ns, hv.y));
    if (bias != nullptr) {
      acc.x = __fadd_rn(acc.x, bias[2 * lane]);
      acc.y = __fadd_rn(acc.y, bias[2 * lane + 1]);
    }
    if (RELU) {
      acc.x = fmaxf(acc.x, 0.f);
      acc.y = fmaxf(acc.y, 0.f);
    }
    *reinterpret_cast<float2*>(out + i * ldo + 2 * lane) = acc;
  }
}

// ---- backward: a_e = <g[col_e], h[row_e]> per edge, a_self[i] = <g[i], h[i]> -----------------
// half-warp per item (16 lanes x float4), fixed xor tree: deterministic
__global__ void __launch_bounds__(256) k_w_edge_dot(const int64_t* __restrict__ ei, int64_t E, int64_t N,
                                                    const float* __restrict__ g, const float* __restrict__ h,
                                                    float* __restrict__ a_e, float* __restrict__ a_self) {
  const int hl = threadIdx.x & 15;
  const int64_t item0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 4;
  const int64_t nitem = ((int64_t)gridDim.x * blockDim.x) >> 4;
  const int64_t total = (E + N + 1) / 2 * 2;   // both halves of a warp stay in the loop together
  for (int64_t it = item0; it < total; it += nitem) {
    int64_t r = -1, c = -1;
    if (it < E) {
      r = ei[it];
      c = ei[E + it];
      if (r == c || r < 0 || r >= N || c < 0 || c >= N) r = c = -1;
    } else if (it < E + N) {
      r = c = it - E;
    }
    float d = 0.f;
    if (r >= 0) {
      const float4 gv = *reinterpret_cast<const float4*>(g + c * H + 4 * hl);
      const float4 hv = *reinterpret_cast<const float4*>(h + r * H + 4 * hl);
      d = gv.x * hv.x + gv.y * hv.y + gv.z * hv.z + gv.w * hv.w;
    }
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) d += __shfl_xor_sync(FULL_MASK, d, o);
    if (hl == 0) {
      if (it < E) a_e[it] = d;
      else if (it < E + N) a_self[it - E] = d;
    }
  }
}

// ---- backward: dL/ddeg[j] = -1/2 dis_j^3 * dL/ddis_j,
//      dL/ddis_j = sum_{e: row=j} (w_e dis[col]) a_e + sum_{e: col=j} (dis[row] w_e) a_e + 2 self_w_j dis_j a_self_j
// direction blockIdx.y of `a` (one launch for both directions of the feature path)
__global__ void __launch_bounds__(256) k_w_ddeg(WGradArgs a) {
  const WGradDir& p = a.d[blockIdx.y];
  if (p.dw == nullptr) return;
  const WGraph& G = p.G;
  const float* __restrict__ w = p.w;
  const float* __restrict__ a_e = p.a_e;
  const int64_t N = a.N;
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarp = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t j = warp0; j < N; j += nwarp) {
    float acc = 0.f;
    for (int o = 0; o < 2; ++o) {
      const int32_t* ptr = o ? G.g.in_ptr : G.g.out_ptr;
      const int32_t* idx = o ? G.g.in_idx : G.g.out_idx;
      const int32_t* eid = o ? G.in_eid : G.out_eid;
      const int s = ptr[j], e = ptr[j + 1];
      for (int b = s; b < e; b += 32) {
        const int n = min(32, e - b);
        float q = 0.f;
        if (lane < n) {
          const int ed = eid[b + lane];
          q = G.dis[idx[b + lane]] * w[ed] * a_e[ed];
        }
        for (int l = 0; l < n; ++l) acc += __shfl_sync(FULL_MASK, q, l);
      }
    }
    const float dj = G.dis[j];
    acc += 2.f * G.self_w[j] * dj * p.a_self[j];
    if (lane == 0) p.ddeg[j] = -0.5f * dj * dj * dj * acc;
  }
}

// ---- backward: gradient of every edge weight (direction blockIdx.y) ---------------------------
__global__ void k_w_dweight(WGradArgs a) {
  const WGradDir& p = a.d[blockIdx.y];
  if (p.dw == nullptr) return;
  const WGraph& G = p.G;
  const int64_t N = a.N, E = p.E;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = p.ei[e], c = p.ei[E + e];
    float d = 0.f;
    if (r >= 0 && r < N && c >= 0 && c < N) {
      if (r != c) {
        d = G.dis[r] * G.dis[c] * p.a_e[e] + p.ddeg[a.deg_by_source ? r : c];
      } else {
        // a self-loop edge: its weight became self_w[r].  Autograd of the reference's
        // `loop_weight[row[inv]] = edge_weight[inv]` hands the slot's gradient to EVERY loop edge on
        // the node, also the overwritten ones; mirrored here.
        d = G.dis[r] * G.dis[r] * p.a_self[r] + p.ddeg[r];
      }
    }
    p.dw[e] = d;
  }
}

// ---- backward: dx = T W  ([N,64] x [64,K]) -----------------------------------------------------
// thread per output column, 32 rows per CTA held in registers; T tile in shared memory (broadcast
// reads), W streamed coalesced (L2-resident across row tiles), stores coalesced.
constexpr int DX_ROWS = 32;
__global__ void __launch_bounds__(256) k_w_dx(const float* __restrict__ t, const float* __restrict__ w, int64_t ldw,
                                              int64_t N, int64_t K, float* __restrict__ dx, int64_t lddx) {
  __shared__ float ts[DX_ROWS][H];
  const int64_t row0 = (int64_t)blockIdx.y * DX_ROWS;
  for (int i = threadIdx.x; i < DX_ROWS * H; i += 256) {
    const int64_t r = row0 + i / H;
    ts[i / H][i % H] = r < N ? t[r * H + i % H] : 0.f;
  }
  __syncthreads();
  const int64_t k = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (k >= K) return;
  float acc[DX_ROWS];
#pragma unroll
  for (int r = 0; r < DX_ROWS; ++r) acc[r] = 0.f;
#pragma unroll 4
  for (int o = 0; o < H; ++o) {
    const float wv = w[(int64_t)o * ldw + k];
#pragma unroll
    for (int r = 0; r < DX_ROWS; ++r) acc[r] = fmaf(ts[r][o], wv, acc[r]);
  }
#pragma unroll
  for (int r = 0; r < DX_ROWS; ++r)
    if (row0 + r < N) dx[(row0 + r) * lddx + k] = acc[r];
}

// ---- host side ---------------------------------------------------------------------------------
static int grid_for(int64_t work_items, int per_block) {
  int64_t b = ceil_div(work_items > 0 ? work_items : 1, per_block);
  const int64_t cap = (int64_t)num_sms() * 8;
  return (int)(b > cap ? cap : b);
}

struct WNormWs {
  WGraph G;
  void* prep_ws; size_t prep_bytes;
};
static void carve_wnorm(Carver& c, int64_t N, int64_t E, WNormWs& w, bool own_outputs, float* norm_e, float* norm_self,
                        float* dis) {
  const size_t n1 = (size_t)(N > 0 ? N : 1), e1 = (size_t)(E > 0 ? E : 1);
  w.G.g.in_ptr = c.take<int32_t>(N + 1);
  w.G.g.out_ptr = c.take<int32_t>(N + 1);
  w.G.g.in_idx = c.take<int32_t>(e1);
  w.G.g.out_idx = c.take<int32_t>(e1);
  w.G.g.deg = c.take<int32_t>(n1);
  w.G.g.dis = c.take<float>(n1);
  w.G.g.rowsum = nullptr;
  w.G.g.in_long = nullptr;
  w.G.g.out_long = nullptr;
  w.G.in_eid = c.take<int32_t>(e1);
  w.G.out_eid = c.take<int32_t>(e1);
  w.G.loop_eid = c.take<int32_t>(n1);
  w.G.self_w = c.take<float>(n1);
  w.G.dis = own_outputs ? c.take<float>(n1) : dis;
  w.G.norm_e = own_outputs ? c.take<float>(e1) : norm_e;
  w.G.norm_self = own_outputs ? c.take<float>(n1) : norm_self;
  w.prep_bytes = graph_prep_ws_bytes(N, E, 1);
  w.prep_ws = c.take<char>(w.prep_bytes);
}

static int wnorm_run(const WNormWs& w, const int64_t* edge_index, int64_t E, const float* edge_weight, int64_t N,
                     int32_t deg_by, int32_t* flags, cudaStream_t st) {
  const int64_t* ei[1] = {edge_index};
  const int64_t Es[1] = {E};
  int32_t* eids[2] = {w.G.in_eid, w.G.out_eid};
  if (int rc = graph_prep_impl(1, ei, Es, N, nullptr, 0, deg_by, &w.G.g, nullptr, flags, w.prep_ws, w.prep_bytes, st,
                               eids))
    return rc;
  if (N == 0) return 0;
  cudaMemsetAsync(w.G.loop_eid, 0xFF, (size_t)N * sizeof(int32_t), st);
  if (E > 0) {
    k_w_loops<<<grid_for(E, 256), 256, 0, st>>>(edge_index, E, N, w.G.loop_eid);
    BIGCN_CHECK_LAUNCH("k_w_loops");
  }
  k_w_deg<<<grid_for(N, 8), 256, 0, st>>>(w.G, edge_weight, N, deg_by == BIGCN_DEG_BY_SOURCE);
  BIGCN_CHECK_LAUNCH("k_w_deg");
  if (E > 0) {
    k_w_norm<<<grid_for(E, 256), 256, 0, st>>>(w.G, edge_index, edge_weight, E, N);
    BIGCN_CHECK_LAUNCH("k_w_norm");
  }
  return 0;
}

struct WConvWs {
  WNormWs n;
  float* wT;       // [K][128] transposed weight / TF32 split scratch of xw_dispatch
  float* xw;       // [N][64]  h = x W^T (kept for the edge-weight gradient)
  float* t;        // [N][64]  T = A-hat^T grad_out
  float* split;    // [2][N][64]
  float* a_e;      // [E]
  float* a_self;   // [N]
  float* ddeg;     // [N]
  float* cs_part;
  float* dw_part;
  size_t total;
};
static WConvWs carve_wconv(int64_t N, int64_t E, int64_t K, void* ws, size_t bytes) {
  WConvWs w{};
  Carver c(ws, bytes);
  const size_t n1 = (size_t)(N > 0 ? N : 1), e1 = (size_t)(E > 0 ? E : 1);
  carve_wnorm(c, N, E, w.n, true, nullptr, nullptr, nullptr);
  w.wT = c.take<float>((size_t)K * H * 2);
  w.xw = c.take<float>(n1 * H);
  w.t = c.take<float>(n1 * H);
  w.split = c.take<float>(n1 * H * 2);
  w.a_e = c.take<float>(e1);
  w.a_self = c.take<float>(n1);
  w.ddeg = c.take<float>(n1);
  w.cs_part = c.take<float>((size_t)cs_chunks(N) * H);
  w.dw_part = c.take<float>(dw_partial_floats(N, K, 64));
  w.total = align_up(c.off, 256);
  return w;
}

// ---- the two-direction feature path on an edge-weighted batch (api.cu) -------------------------------------------
// The feature path's own graph prep runs with the edge id as the sort payload; on top of it, per direction, the
// normalisation above (k_w_loops, k_w_deg, k_w_norm) and then the normalised weights laid out in both CSR orders for
// the tuned sweeps of gather.cuh (WtEntry): in_w[k] = norm_e[in_eid[k]] (A-hat), out_w[k] = norm_e[out_eid[k]]
// (A-hat^T); the self-loop weights are norm_self.  With every weight 1 these are (dis[j] * 1) * dis[i] = dis[j] * dis[i]
// and (dis[i] * 1) * dis[i], and the degree is a float sum of ones: the unweighted values, bit for bit.
__global__ void k_wf_entries(WGraph G, const float* __restrict__ w, int64_t E, int64_t N, float* __restrict__ in_w,
                             float* __restrict__ out_w, int32_t* flags) {
  bool bad = false;
  const int64_t n = E > N ? E : N;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
    if (t < E) {
      in_w[t] = G.norm_e[G.in_eid[t]];
      out_w[t] = G.norm_e[G.out_eid[t]];
      bad |= !isfinite(w[t]);
    }
    if (t < N) bad |= isnan(G.dis[t]);   // a negative weighted degree
  }
  if (bad) atomicOr(flags, BIGCN_FLAG_EDGE_WEIGHT);
}

__global__ void k_wf_fill(float* __restrict__ p, int64_t n, float v) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) p[t] = v;
}

int wfeat_ones(float* ones, int64_t n, cudaStream_t st) {
  if (n <= 0) return 0;
  k_wf_fill<<<grid_for(n, 256), 256, 0, st>>>(ones, n, 1.0f);
  BIGCN_CHECK_LAUNCH("k_wf_fill");
  return 0;
}

int wfeat_prep(const WGraph& G, const int64_t* ei, int64_t E, const float* w, int64_t N, int32_t deg_by, float* in_w,
               float* out_w, int32_t* flags, cudaStream_t st) {
  if (N == 0) return 0;
  cudaMemsetAsync(G.loop_eid, 0xFF, (size_t)N * sizeof(int32_t), st);
  if (E > 0) {
    k_w_loops<<<grid_for(E, 256), 256, 0, st>>>(ei, E, N, G.loop_eid);
    BIGCN_CHECK_LAUNCH("k_w_loops");
  }
  k_w_deg<<<grid_for(N, 8), 256, 0, st>>>(G, w, N, deg_by == BIGCN_DEG_BY_SOURCE);
  BIGCN_CHECK_LAUNCH("k_w_deg");
  if (E > 0) {
    k_w_norm<<<grid_for(E, 256), 256, 0, st>>>(G, ei, w, E, N);
    BIGCN_CHECK_LAUNCH("k_w_norm");
  }
  k_wf_entries<<<grid_for(E > N ? E : N, 256), 256, 0, st>>>(G, w, E, N, in_w, out_w, flags);
  BIGCN_CHECK_LAUNCH("k_wf_entries");
  return 0;
}

// ---- edge gradient of the feature path: both convs of a direction share the edge list, so
//   a_e    = <G1[c], XW[r]> + <G2[c], M[r]>   for edge e = (r -> c), 0 for self-loop / out-of-range edges
//   a_self = the same with r = c = i
// with G1 the gradient at conv1's output, XW conv1's propagate input, M conv2's (the mix kernel's z) and
// G2[c] = [H2[c] > 0] * gs[batch[c]] formed here as k_propagate_g2 forms it.  The rest of the chain (through dis and
// the self-loop weights) is k_w_ddeg / k_w_dweight above.  Half-warp per item, each lane adds its four conv1 products,
// then its four conv2 products, then the two; a fixed xor tree across the 16 lanes: deterministic, no atomics.
__global__ void __launch_bounds__(256) k_wf_edge_dot(EdgeDotArgs a) {
  const EdgeDotDir& p = a.d[blockIdx.y];
  if (p.a_e == nullptr) return;
  const int hl = threadIdx.x & 15;
  const int64_t N = a.N, E = p.E;
  const int64_t item0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 4;
  const int64_t nitem = ((int64_t)gridDim.x * blockDim.x) >> 4;
  const int64_t total = (E + N + 1) / 2 * 2;   // both halves of a warp stay in the loop together
  for (int64_t it = item0; it < total; it += nitem) {
    int64_t r = -1, c = -1;
    if (it < E) {
      r = p.ei[it];
      c = p.ei[E + it];
      if (r == c || r < 0 || r >= N || c < 0 || c >= N) r = c = -1;
    } else if (it < E + N) {
      r = c = it - E;
    }
    float d = 0.f;
    if (r >= 0) {
      const float4 g1 = *reinterpret_cast<const float4*>(p.g1 + c * H + 4 * hl);
      const float4 xw = *reinterpret_cast<const float4*>(p.xw + r * p.ldxw + 4 * hl);
      const float4 h2 = *reinterpret_cast<const float4*>(p.h2 + c * H + 4 * hl);
      const float4 gs = *reinterpret_cast<const float4*>(p.gs + a.batch[c] * H + 4 * hl);
      const float4 m = *reinterpret_cast<const float4*>(p.m + r * H + 4 * hl);
      const float d1 = g1.x * xw.x + g1.y * xw.y + g1.z * xw.z + g1.w * xw.w;
      const float d2 = (h2.x > 0.f ? gs.x : 0.f) * m.x + (h2.y > 0.f ? gs.y : 0.f) * m.y +
                       (h2.z > 0.f ? gs.z : 0.f) * m.z + (h2.w > 0.f ? gs.w : 0.f) * m.w;
      d = d1 + d2;
    }
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) d += __shfl_xor_sync(FULL_MASK, d, o);
    if (hl == 0) {
      if (it < E) p.a_e[it] = d;
      else if (it < E + N) p.a_self[it - E] = d;
    }
  }
}

int wfeat_edge_dot(const EdgeDotArgs& a, int ndir, cudaStream_t st) {
  int64_t m = 0;
  for (int q = 0; q < ndir; ++q)
    if (a.d[q].a_e && a.d[q].E + a.N > m) m = a.d[q].E + a.N;
  if (m == 0) return 0;
  k_wf_edge_dot<<<dim3(grid_for(m, 16), ndir), 256, 0, st>>>(a);
  BIGCN_CHECK_LAUNCH("k_wf_edge_dot");
  return 0;
}

int wfeat_edge_grad(const WGradArgs& a, int ndir, cudaStream_t st) {
  int64_t emax = 0;
  bool any = false;
  for (int q = 0; q < ndir; ++q) {
    if (a.d[q].dw == nullptr) continue;
    any = true;
    if (a.d[q].E > emax) emax = a.d[q].E;
  }
  if (!any) return 0;
  if (a.N > 0) {
    k_w_ddeg<<<dim3(grid_for(a.N, 8), ndir), 256, 0, st>>>(a);
    BIGCN_CHECK_LAUNCH("k_w_ddeg");
  }
  if (emax > 0) {
    k_w_dweight<<<dim3(grid_for(emax, 256), ndir), 256, 0, st>>>(a);
    BIGCN_CHECK_LAUNCH("k_w_dweight");
  }
  return 0;
}

int w_propagate_launch(const int32_t* ptr, const int32_t* idx, const int32_t* eid, const float* norm_e,
                       const float* norm_self, const float* h, const float* bias, float* out, int64_t N, bool relu,
                       cudaStream_t st) {
  if (N == 0) return 0;
  if (relu) k_w_propagate<true><<<grid_for(N, 8), 256, 0, st>>>(ptr, idx, eid, norm_e, norm_self, h, H, bias, out, H, N);
  else k_w_propagate<false><<<grid_for(N, 8), 256, 0, st>>>(ptr, idx, eid, norm_e, norm_self, h, H, bias, out, H, N);
  BIGCN_CHECK_LAUNCH("k_w_propagate");
  return 0;
}

int w_edge_dot_launch(const int64_t* ei, int64_t E, int64_t N, const float* g, const float* h, float* a_e, float* a_self,
                      cudaStream_t st) {
  if (N == 0) return 0;
  k_w_edge_dot<<<grid_for(E + N, 16), 256, 0, st>>>(ei, E, N, g, h, a_e, a_self);
  BIGCN_CHECK_LAUNCH("k_w_edge_dot");
  return 0;
}

}  // namespace bigcn

using namespace bigcn;

extern "C" size_t bigcn_gcn_norm_weighted_workspace_bytes(int64_t N, int64_t E) {
  WNormWs w{};
  Carver c(nullptr, 0);
  carve_wnorm(c, N, E, w, false, nullptr, nullptr, nullptr);
  return align_up(c.off, 256);
}

extern "C" int bigcn_gcn_norm_weighted(const int64_t* edge_index, int64_t E, const float* edge_weight, int64_t N,
                                       int32_t deg_by, float* norm_e, float* norm_self, float* dis, int32_t* flags,
                                       void* workspace, size_t workspace_bytes, bigcn_stream_t stream) {
  BIGCN_CHECK_ARG(N >= 0 && E >= 0 && flags && (E == 0 || (edge_index && edge_weight && norm_e)) &&
                      (N == 0 || (norm_self && dis)), "gcn_norm_weighted: bad arguments");
  WNormWs w{};
  Carver c(workspace, workspace_bytes);
  carve_wnorm(c, N, E, w, false, norm_e, norm_self, dis);
  BIGCN_CHECK_ARG(workspace && c.ok(), "gcn_norm_weighted: workspace too small");
  return wnorm_run(w, edge_index, E, edge_weight, N, deg_by, flags, (cudaStream_t)stream);
}

extern "C" size_t bigcn_gcnconv_weighted_workspace_bytes(int64_t N, int64_t E, int64_t K) {
  return carve_wconv(N, E, K, nullptr, 0).total;
}

extern "C" int bigcn_gcnconv_weighted_forward(const float* x, int64_t N, int64_t K, const int64_t* edge_index, int64_t E,
                                              const float* edge_weight, const float* w, const float* bias,
                                              int32_t deg_by, int32_t gemm_mode, float* out, int32_t* flags,
                                              void* workspace, size_t workspace_bytes, bigcn_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  BIGCN_CHECK_ARG(N >= 0 && K > 0 && E >= 0 && w && flags && (E == 0 || (edge_index && edge_weight)),
                  "gcnconv_weighted_forward: bad arguments");
  BIGCN_CHECK_ARG(gemm_mode != BIGCN_GEMM_BF16, "gcnconv_weighted_forward: gemm_mode BF16 is not supported here (fp32 x)");
  WConvWs cw = carve_wconv(N, E, K, workspace, workspace_bytes);
  BIGCN_CHECK_ARG(workspace && workspace_bytes >= cw.total, "gcnconv_weighted_forward: workspace too small");
  if (int rc = wnorm_run(cw.n, edge_index, E, edge_weight, N, deg_by, flags, st)) return rc;
  if (N == 0) return 0;
  BIGCN_CHECK_ARG(x && out, "gcnconv_weighted_forward: NULL argument");
  const float* ws1[1] = {w};
  if (int rc = xw_dispatch(x, N, K, ws1, 1, K, cw.wT, cw.xw, H, gemm_mode, st)) return rc;
  const WGraph& G = cw.n.G;
  k_w_propagate<false><<<grid_for(N, 8), 256, 0, st>>>(G.g.in_ptr, G.g.in_idx, G.in_eid, G.norm_e, G.norm_self, cw.xw, H, bias,
                                                out, H, N);
  BIGCN_CHECK_LAUNCH("k_w_propagate");
  return 0;
}

extern "C" int bigcn_gcnconv_weighted_backward(const float* x, int64_t N, int64_t K, const int64_t* edge_index, int64_t E,
                                               const float* edge_weight, const float* w, const float* grad_out,
                                               float* dw, float* db, float* d_edge_weight, float* dx, int32_t deg_by,
                                               int32_t gemm_mode, void* workspace, size_t workspace_bytes,
                                               bigcn_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  BIGCN_CHECK_ARG(N >= 0 && K > 0 && E >= 0 && dw && db, "gcnconv_weighted_backward: bad arguments");
  BIGCN_CHECK_ARG(gemm_mode != BIGCN_GEMM_BF16, "gcnconv_weighted_backward: gemm_mode BF16 is not supported here (fp32 x)");
  WConvWs cw = carve_wconv(N, E, K, workspace, workspace_bytes);
  BIGCN_CHECK_ARG(workspace && workspace_bytes >= cw.total, "gcnconv_weighted_backward: workspace too small");
  const WGraph& G = cw.n.G;
  if (int rc = colsum64_launch(grad_out, N, cw.cs_part, db, st)) return rc;
  if (N > 0) {
    // T = A-hat^T grad_out: the by-source CSR with the same per-edge norms
    k_w_propagate<false><<<grid_for(N, 8), 256, 0, st>>>(G.g.out_ptr, G.g.out_idx, G.out_eid, G.norm_e, G.norm_self, grad_out,
                                                  H, nullptr, cw.t, H, N);
    BIGCN_CHECK_LAUNCH("k_w_propagate");
  }
  if (d_edge_weight != nullptr && N > 0) {
    k_w_edge_dot<<<grid_for(E + N, 16), 256, 0, st>>>(edge_index, E, N, grad_out, cw.xw, cw.a_e, cw.a_self);
    BIGCN_CHECK_LAUNCH("k_w_edge_dot");
    WGradArgs ga{};
    ga.d[0] = WGradDir{G, edge_index, E, edge_weight, cw.a_e, cw.a_self, cw.ddeg, d_edge_weight};
    ga.N = N; ga.deg_by_source = deg_by == BIGCN_DEG_BY_SOURCE;
    if (int rc = wfeat_edge_grad(ga, 1, st)) return rc;
  } else if (d_edge_weight != nullptr && E > 0) {
    cudaMemsetAsync(d_edge_weight, 0, (size_t)E * sizeof(float), st);
  }
  if (dx != nullptr && N > 0) {
    BIGCN_CHECK_ARG(w != nullptr, "gcnconv_weighted_backward: dx needs the weight");
    BIGCN_CHECK_ARG(ceil_div(N, DX_ROWS) <= 65535, "gcnconv_weighted_backward: dx supports N <= %d", 65535 * DX_ROWS);
    k_w_dx<<<dim3((unsigned)ceil_div(K, 256), (unsigned)ceil_div(N, DX_ROWS)), 256, 0, st>>>(cw.t, w, K, N, K, dx, K);
    BIGCN_CHECK_LAUNCH("k_w_dx");
  }
  // dw = T^T x
  if (gemm_mode == BIGCN_GEMM_SPARSE) gemm_mode = BIGCN_GEMM_FP32;
  if (gemm_mode == BIGCN_GEMM_FP32) return dw_fp32(x, N, K, cw.t, H, 64, cw.dw_part, dw, K, 0, nullptr, 0, 0, st);
  return dw_tc(x, N, K, cw.t, H, 64, cw.split, cw.split + (size_t)(N > 0 ? N : 1) * H, cw.dw_part, dw, K, 0, nullptr, 0,
               0, gemm_mode, st);
}
