// EBGCN's second conv (model/Twitter/EBGCN.py:71-85, BU twin :168-182) for one direction:
//
//   root_extend = x[rootindex[batch]]                      N x K
//   u = relu(bn1(cat(h1, root_extend)))                    N x (64 + K)
//   out = relu(conv2(u, edge_index, edge_weight))          N x 64
//
// without forming anything N x K.  Every row of root_extend in tree b is x[r_b], so with n_b the size of tree b the batch
// statistics of the K root columns are count-weighted statistics over B root rows (two passes, mean first):
//   mu_k = sum_b n_b x[r_b,k] / N,   var_k = sum_b n_b (x[r_b,k] - mu_k)^2 / N
// the normalised, relu'd root half is one row per tree, R_b = relu(gamma (x[r_b] - mu) / sqrt(var + eps) + beta) [B,K],
// and so is its conv2 product, Y_b = R_b W2b^T [B,64].  Per node Z_i = relu(bn(h1_i)) W2a^T + Y_b(i); then the weighted
// propagate of weighted.cu (gcn_norm with weights, per-row sums in edge-list order) adds b2 and applies the relu.
//
// Backward from G = grad_out * [out > 0]: T = A-hat^T G, S_b = sum_{i in b} T_i (k_segsum), dW2a = T^T A (k_outer64),
// dW2b = S^T R (the dW scan of xw.cu over R), dR = (S W2b) [R > 0] -> dbeta_k = sum_b dR_bk, dgamma_k = sum_b dR_bk xhat_bk
// (k_eb_root_bwd), and for the 64 h1 columns an ordinary BatchNorm backward over N rows (k_eb_hbwd1 / k_eb_hbwd2).
// d edge_weight: the chain of weighted.cu (k_w_edge_dot with Z as the propagated operand, k_w_ddeg, k_w_dweight).
// A CSR x (bigcn_ebgcn_t.x == NULL) is read at the roots only: k_eb_root_csr fills a dense block Xr [B,K] of the B root
// rows and a tree-local root map, and the kernels below run unchanged on Xr with that map (r_b = b).
// Every reduction runs in a fixed order (row / tree segments combined in index order): deterministic, no atomics on
// floats.  bn1's sums over N rows (statistics, dbeta, dgamma) accumulate in fp64: BatchNorm's output is centred, so a
// shift of the mean by a few fp32 ulps of its partial sums enters every row's term of dW2 = T^T A with the same sign.
#include "kernels.cuh"

namespace bigcn {

constexpr int EB_ROWS = 128;   // node rows per CTA of the h1-column kernels (8 warps x 16 rows)
constexpr int EB_TREES = 32;   // trees per segment of the root-column reductions

struct Eb {
  int64_t N, B, K, ld;          // ld = 64 + K, the row pitch of W2
  const float* h1; const float* x; const int64_t* batch; const int32_t* root; const int32_t* node_ptr;
  const float* gamma; const float* beta;   // NULL: no affine (or bn1 skipped)
  float* mean; float* invstd;   // [64 + K]: the statistics that normalise (batch or running)
  double* meand;                // [64 + K]: the batch mean in fp64 (the second statistics pass)
  double* hpart;                // [nh][128] h1-column partials
  double* rpart;                // [nseg][2K] root-column partials
  int32_t nh, nseg;
  float* rm; float* rv; int64_t* nbt;
  float momentum, eps;
  int32_t update;               // training with running statistics
  const float* w2;
  float* R; const float* Y; float* A; float* Z;
  const float* T; const float* S; float* G; double* dgb;  // dgb [2][64]: dbeta, dgamma of the h1 columns
};

__device__ __forceinline__ float eb_bn(const Eb& a, float v, int64_t c) {
  const float y = (v - a.mean[c]) * a.invstd[c];
  return a.gamma != nullptr ? fmaf(y, a.gamma[c], a.beta[c]) : y;
}

// root row of every non-empty tree (-1: empty tree, or an out-of-range rootindex, which is flagged)
__global__ void k_eb_roots(const int64_t* __restrict__ rootindex, const int32_t* __restrict__ node_ptr, int64_t B,
                           int64_t N, int32_t* __restrict__ root, int32_t* flags) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const bool nonempty = node_ptr[b + 1] > node_ptr[b];
  const int64_t r = rootindex[b];
  const bool ok = r >= 0 && r < N;
  if (nonempty && !ok) atomicOr(flags, BIGCN_FLAG_ROOT_RANGE);
  root[b] = nonempty && ok ? (int32_t)r : -1;
}

// CSR x: Xr[b] = x[r_b] as a dense row (zeroed, then the row's entries added in CSR order; a column outside [0, K) is
// skipped and flagged), rmap[b] = b, or -1 where root[b] is -1 (Xr[b] then stays zero).  CTA per tree.
__global__ void __launch_bounds__(128) k_eb_root_csr(const int32_t* __restrict__ root, const int32_t* __restrict__ ptr,
                                                     const int32_t* __restrict__ col, const float* __restrict__ val,
                                                     int64_t K, float* __restrict__ Xr, int32_t* __restrict__ rmap,
                                                     int32_t* flags) {
  const int64_t b = blockIdx.x;
  const int32_t r = root[b];
  float* row = Xr + b * K;
  for (int64_t k = threadIdx.x; k < K; k += blockDim.x) row[k] = 0.f;
  if (threadIdx.x == 0) rmap[b] = r >= 0 ? (int32_t)b : -1;
  if (r < 0) return;   // the same for the whole CTA
  __syncthreads();
  if (threadIdx.x != 0) return;
  const int p1 = ptr[r + 1];
  for (int p = ptr[r]; p < p1; ++p) {
    const int k = col[p];
    if (k < 0 || k >= K) {
      atomicOr(flags, BIGCN_FLAG_X_CSR_RANGE);
      continue;
    }
    row[k] += val[p];
  }
}

// ---- bn1 statistics: PASS 0 sums the values, PASS 1 the squared deviations from the mean of PASS 0 -----------------
// h1 columns: CTA = EB_ROWS rows, 4 row groups x 64 columns, groups combined in order
template <int PASS>
__global__ void __launch_bounds__(256) k_eb_hstat(Eb a) {
  __shared__ double red[4][H];
  const int g = threadIdx.x >> 6, c = threadIdx.x & 63;
  const int64_t i0 = (int64_t)blockIdx.x * EB_ROWS, i1 = min(a.N, i0 + EB_ROWS);
  const double mu = PASS ? a.meand[c] : 0.0;
  double s = 0.0;
  for (int64_t i = i0 + g; i < i1; i += 4) {
    const double v = a.h1[i * H + c];
    if (PASS) {
      const double d = v - mu;
      s = fma(d, d, s);
    } else {
      s += v;
    }
  }
  red[g][c] = s;
  __syncthreads();
  if (g == 0) a.hpart[(int64_t)blockIdx.x * 2 * H + c] = ((red[0][c] + red[1][c]) + red[2][c]) + red[3][c];
}

// root columns: thread per column, the EB_TREES trees of segment blockIdx.y in order, each weighted by its node count
template <int PASS>
__global__ void __launch_bounds__(256) k_eb_rstat(Eb a) {
  const int64_t k = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (k >= a.K) return;
  const int64_t b0 = (int64_t)blockIdx.y * EB_TREES, b1 = min(a.B, b0 + EB_TREES);
  const double mu = PASS ? a.meand[H + k] : 0.0;
  double s = 0.0;
  for (int64_t b = b0; b < b1; ++b) {
    const int32_t r = a.root[b];
    if (r < 0) continue;
    const double n = (double)(a.node_ptr[b + 1] - a.node_ptr[b]);
    const double v = a.x[(int64_t)r * a.K + k];
    if (PASS) {
      const double d = v - mu;
      s = fma(n, d * d, s);
    } else {
      s = fma(n, v, s);
    }
  }
  a.rpart[(int64_t)blockIdx.y * 2 * a.K + k] = s;
}

// mode 0: mean (and num_batches_tracked += 1 in training); mode 1: biased variance -> invstd, running statistics
// moved (torch: running = f * batch + (1 - f) * running, unbiased variance, f = 1 / num_batches_tracked for
// momentum=None); mode 2: the running statistics normalise; mode 3: bn1 skipped (mean 0, invstd 1: the identity)
__global__ void __launch_bounds__(256) k_eb_stat_fin(Eb a, int mode) {
  const int64_t c = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (mode == 0 && c == 0 && a.update && a.nbt != nullptr) a.nbt[0] += 1;
  if (c >= H + a.K) return;
  if (mode >= 2) {
    a.mean[c] = mode == 2 ? a.rm[c] : 0.f;
    a.invstd[c] = mode == 2 ? 1.f / sqrtf(a.rv[c] + a.eps) : 1.f;
    return;
  }
  double s = 0.0;
  if (c < H) {
    for (int j = 0; j < a.nh; ++j) s += a.hpart[(int64_t)j * 2 * H + c];
  } else {
    for (int j = 0; j < a.nseg; ++j) s += a.rpart[(int64_t)j * 2 * a.K + c - H];
  }
  const double n = (double)a.N;
  if (mode == 0) {
    a.meand[c] = s / n;
    a.mean[c] = (float)(s / n);
    return;
  }
  const double var = s / n;
  a.invstd[c] = (float)(1.0 / sqrt(var + (double)a.eps));
  if (a.update) {
    const float f = a.momentum < 0.f ? (float)(1.0 / (double)a.nbt[0]) : a.momentum;
    a.rm[c] = f * a.mean[c] + (1.f - f) * a.rm[c];
    a.rv[c] = f * (float)(var * n / (n - 1.0)) + (1.f - f) * a.rv[c];
  }
}

// R[b][k] = relu(bn1(x[r_b][k])) for column 64 + k (0 for an empty tree)
__global__ void __launch_bounds__(256) k_eb_root_r(Eb a) {
  const int64_t total = a.B * a.K;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = t / a.K, k = t - b * a.K;
    const int32_t r = a.root[b];
    a.R[t] = r >= 0 ? fmaxf(eb_bn(a, a.x[(int64_t)r * a.K + k], H + k), 0.f) : 0.f;
  }
}

// A_i = relu(bn1(h1_i)), Z_i = A_i W2a^T + Y_b(i): warp per row, lane owns outputs lane and lane + 32, W2a^T in shared
// memory, the row's A broadcast from shared memory, columns ascending
__global__ void __launch_bounds__(256) k_eb_mix(Eb a) {
  __shared__ float sW[H][H + 1];   // sW[c][o] = W2[o][c]
  __shared__ float sA[8][H];
  for (int t = threadIdx.x; t < H * H; t += 256) sW[t & 63][t >> 6] = a.w2[(int64_t)(t >> 6) * a.ld + (t & 63)];
  __syncthreads();
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t base = (int64_t)blockIdx.x * EB_ROWS + w * 16;
  for (int rr = 0; rr < 16; ++rr) {
    const int64_t i = base + rr;
    if (i >= a.N) break;
    const float a0 = fmaxf(eb_bn(a, a.h1[i * H + lane], lane), 0.f);
    const float a1 = fmaxf(eb_bn(a, a.h1[i * H + lane + 32], lane + 32), 0.f);
    a.A[i * H + lane] = a0;
    a.A[i * H + lane + 32] = a1;
    sA[w][lane] = a0;
    sA[w][lane + 32] = a1;
    __syncwarp();
    float z0 = 0.f, z1 = 0.f;
#pragma unroll 16
    for (int c = 0; c < H; ++c) {
      const float av = sA[w][c];
      z0 = fmaf(av, sW[c][lane], z0);
      z1 = fmaf(av, sW[c][lane + 32], z1);
    }
    __syncwarp();
    const int64_t b = a.batch[i];
    if (b >= 0 && b < a.B) {
      z0 += a.Y[b * H + lane];
      z1 += a.Y[b * H + lane + 32];
    }
    a.Z[i * H + lane] = z0;
    a.Z[i * H + lane + 32] = z1;
  }
}

// ---- backward --------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_eb_gmask(const float* __restrict__ g, const float* __restrict__ out, int64_t n,
                                                   float* __restrict__ gm) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x)
    gm[t] = out[t] > 0.f ? g[t] : 0.f;
}

// root columns: thread per column k with W2b[:, k] in registers, the trees of segment blockIdx.y in order:
//   dR_bk = [R_bk > 0] sum_o S[b][o] W2[o][64 + k];  dbeta_k += dR_bk;  dgamma_k += dR_bk xhat_bk
__global__ void __launch_bounds__(128) k_eb_root_bwd(Eb a) {
  __shared__ float sS[EB_TREES][H];
  const int64_t b0 = (int64_t)blockIdx.y * EB_TREES, b1 = min(a.B, b0 + EB_TREES);
  for (int t = threadIdx.x; t < EB_TREES * H; t += 128) {
    const int64_t b = b0 + (t >> 6);
    sS[t >> 6][t & 63] = b < b1 ? a.S[b * H + (t & 63)] : 0.f;
  }
  __syncthreads();
  const int64_t k = (int64_t)blockIdx.x * 128 + threadIdx.x;
  if (k >= a.K) return;
  float wk[H];
#pragma unroll
  for (int o = 0; o < H; ++o) wk[o] = a.w2[(int64_t)o * a.ld + H + k];
  const float mu = a.mean[H + k], is = a.invstd[H + k];
  double db = 0.0, dg = 0.0;
  for (int64_t b = b0; b < b1; ++b) {
    const int32_t r = a.root[b];
    if (r < 0 || !(a.R[b * a.K + k] > 0.f)) continue;
    const float* s = sS[b - b0];
    float d = 0.f;
#pragma unroll
    for (int o = 0; o < H; ++o) d = fmaf(s[o], wk[o], d);
    const float xh = (a.x[(int64_t)r * a.K + k] - mu) * is;
    db += d;
    dg = fma((double)d, (double)xh, dg);
  }
  a.rpart[(int64_t)blockIdx.y * 2 * a.K + k] = db;
  a.rpart[(int64_t)blockIdx.y * 2 * a.K + a.K + k] = dg;
}

// h1 columns, pass 1: G_i = (T_i W2a) [A_i > 0], the gradient at bn1's output; per-CTA column sums of G and G xhat
// (warps combined in order).  Warp per row as in k_eb_mix.
__global__ void __launch_bounds__(256) k_eb_hbwd1(Eb a) {
  __shared__ float sW[H][H + 1];   // sW[o][c] = W2[o][c]
  __shared__ float sT[8][H];
  __shared__ double red[8][2 * H];
  for (int t = threadIdx.x; t < H * H; t += 256) sW[t >> 6][t & 63] = a.w2[(int64_t)(t >> 6) * a.ld + (t & 63)];
  __syncthreads();
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t base = (int64_t)blockIdx.x * EB_ROWS + w * 16;
  const float mu0 = a.mean[lane], mu1 = a.mean[lane + 32], is0 = a.invstd[lane], is1 = a.invstd[lane + 32];
  double sb0 = 0.0, sb1 = 0.0, sg0 = 0.0, sg1 = 0.0;
  for (int rr = 0; rr < 16; ++rr) {
    const int64_t i = base + rr;
    if (i >= a.N) break;
    sT[w][lane] = a.T[i * H + lane];
    sT[w][lane + 32] = a.T[i * H + lane + 32];
    __syncwarp();
    float d0 = 0.f, d1 = 0.f;
#pragma unroll 16
    for (int o = 0; o < H; ++o) {
      const float tv = sT[w][o];
      d0 = fmaf(tv, sW[o][lane], d0);
      d1 = fmaf(tv, sW[o][lane + 32], d1);
    }
    __syncwarp();
    const float g0 = a.A[i * H + lane] > 0.f ? d0 : 0.f;
    const float g1 = a.A[i * H + lane + 32] > 0.f ? d1 : 0.f;
    a.G[i * H + lane] = g0;
    a.G[i * H + lane + 32] = g1;
    sb0 += g0;
    sb1 += g1;
    sg0 = fma((double)g0, (double)((a.h1[i * H + lane] - mu0) * is0), sg0);
    sg1 = fma((double)g1, (double)((a.h1[i * H + lane + 32] - mu1) * is1), sg1);
  }
  red[w][lane] = sb0;
  red[w][lane + 32] = sb1;
  red[w][H + lane] = sg0;
  red[w][H + lane + 32] = sg1;
  __syncthreads();
  if (threadIdx.x < 2 * H) {
    double s = 0.0;
#pragma unroll
    for (int q = 0; q < 8; ++q) s += red[q][threadIdx.x];
    a.hpart[(int64_t)blockIdx.x * 2 * H + threadIdx.x] = s;
  }
}

// dbeta / dgamma of every bn1 column: the partials in order (h1 columns over row chunks, root columns over tree segments)
__global__ void __launch_bounds__(256) k_eb_bwd_fin(Eb a, float* __restrict__ dweight, float* __restrict__ dbias) {
  const int64_t c = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (c >= H + a.K) return;
  double db = 0.0, dg = 0.0;
  if (c < H) {
    for (int j = 0; j < a.nh; ++j) {
      db += a.hpart[(int64_t)j * 2 * H + c];
      dg += a.hpart[(int64_t)j * 2 * H + H + c];
    }
    a.dgb[c] = db;
    a.dgb[H + c] = dg;
  } else {
    for (int j = 0; j < a.nseg; ++j) {
      db += a.rpart[(int64_t)j * 2 * a.K + c - H];
      dg += a.rpart[(int64_t)j * 2 * a.K + a.K + c - H];
    }
  }
  if (dweight != nullptr) dweight[c] = (float)dg;
  if (dbias != nullptr) dbias[c] = (float)db;
}

// h1 columns, pass 2: dh1 = gamma invstd (G - dbeta / N - xhat dgamma / N) with batch statistics (torch's
// batch_norm_backward), gamma invstd G with running statistics, G itself when bn1 is skipped
__global__ void __launch_bounds__(256) k_eb_hbwd2(Eb a, int mode, float* __restrict__ dh1) {
  const int64_t total = a.N * H;
  const double n = (double)a.N;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(t & 63);
    const float g = a.G[t];
    if (mode == 3) {
      dh1[t] = g;
      continue;
    }
    const float is = a.invstd[c], gam = a.gamma != nullptr ? a.gamma[c] : 1.f;
    if (mode == 2) {
      dh1[t] = g * is * gam;
    } else {
      const float xh = (a.h1[t] - a.mean[c]) * is;
      dh1[t] = (g - (float)(a.dgb[c] / n) - xh * (float)(a.dgb[H + c] / n)) * is * gam;
    }
  }
}

// ---- host side -------------------------------------------------------------------------------------------------------
static int eb_grid(int64_t work, int per_block) {
  int64_t b = ceil_div(work > 0 ? work : 1, per_block);
  const int64_t cap = (int64_t)num_sms() * 8;
  return (int)(b > cap ? cap : b);
}

struct EbWs {
  WGraph G;
  void* prep_ws; size_t prep_bytes;
  float* in_w; float* out_w;   // [E] the normalised weights in CSR order (wfeat_prep)
  float* ones;                 // [E] the unit weights of an unweighted conv2
  int32_t* root;               // [B]
  float* mean; float* invstd;  // [64 + K]
  double* meand;               // [64 + K]
  double* hpart;               // [nh][128]
  double* rpart;               // [nseg][2K]
  float* R;                    // [B][K]
  float* Y;                    // [B][64]
  float* wT;                   // [K][64] transposed W2b for the R W2b^T scan
  float* A; float* Z;          // [N][64]
  float* gm;                   // [N][64] grad_out [out > 0], then G
  float* T;                    // [N][64]
  float* S;                    // [B][64]
  float* a_e; float* a_self; float* ddeg;
  float* opart;                // [op_chunks(N)][64 x 64]
  float* dwpart;
  float* cspart;
  double* dgb;                 // [2][64]
  float* Xr;                   // [B][K] CSR x only: the root rows
  int32_t* rmap;               // [B]    CSR x only: b, or -1 for a tree without a root
  int32_t nh, nseg;
  size_t total;
};

static EbWs carve_eb(int64_t N, int64_t B, int64_t K, int64_t E, bool csr, void* ws, size_t bytes) {
  EbWs w{};
  Carver c(ws, bytes);
  const size_t n1 = (size_t)(N > 0 ? N : 1), e1 = (size_t)(E > 0 ? E : 1), b1 = (size_t)(B > 0 ? B : 1);
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
  w.G.dis = c.take<float>(n1);
  w.G.norm_e = c.take<float>(e1);
  w.G.norm_self = c.take<float>(n1);
  w.prep_bytes = graph_prep_ws_bytes(N, E, 1);
  w.prep_ws = c.take<char>(w.prep_bytes);
  w.in_w = c.take<float>(e1);
  w.out_w = c.take<float>(e1);
  w.ones = c.take<float>(e1);
  w.root = c.take<int32_t>(b1);
  w.nh = (int32_t)ceil_div(N > 0 ? N : 1, EB_ROWS);
  w.nseg = (int32_t)ceil_div(B > 0 ? B : 1, EB_TREES);
  w.mean = c.take<float>(H + K);
  w.invstd = c.take<float>(H + K);
  w.meand = c.take<double>(H + K);
  w.hpart = c.take<double>((size_t)w.nh * 2 * H);
  w.rpart = c.take<double>((size_t)w.nseg * 2 * K);
  w.R = c.take<float>(b1 * K);
  w.Y = c.take<float>(b1 * H);
  w.wT = c.take<float>((size_t)K * H);
  w.A = c.take<float>(n1 * H);
  w.Z = c.take<float>(n1 * H);
  w.gm = c.take<float>(n1 * H);
  w.T = c.take<float>(n1 * H);
  w.S = c.take<float>(b1 * H);
  w.a_e = c.take<float>(e1);
  w.a_self = c.take<float>(n1);
  w.ddeg = c.take<float>(n1);
  w.opart = c.take<float>((size_t)op_chunks(N) * H * H);
  w.dwpart = c.take<float>(dw_partial_floats(B, K, H));
  w.cspart = c.take<float>((size_t)cs_chunks(N) * H);
  w.dgb = c.take<double>(2 * H);
  if (csr) {
    w.Xr = c.take<float>(b1 * K);
    w.rmap = c.take<int32_t>(b1);
  }
  w.total = align_up(c.off, 256);
  return w;
}

// 3: bn1 skipped (N == 1), 2: running statistics normalise, 0: batch statistics
static int eb_mode(const bigcn_ebgcn_t* a) {
  if (a->N == 1) return 3;
  return (a->training || a->running_mean == nullptr) ? 0 : 2;
}

static Eb eb_args(const bigcn_ebgcn_t* a, const EbWs& w) {
  Eb e{};
  e.N = a->N; e.B = a->B; e.K = a->K; e.ld = H + a->K;
  e.h1 = a->h1; e.batch = a->batch; e.node_ptr = a->node_ptr;
  e.x = a->x != nullptr ? a->x : w.Xr;
  e.root = a->x != nullptr ? w.root : w.rmap;
  const bool bn = eb_mode(a) != 3;
  e.gamma = bn ? a->bn_weight : nullptr;
  e.beta = bn ? a->bn_bias : nullptr;
  e.mean = w.mean; e.invstd = w.invstd; e.meand = w.meand; e.hpart = w.hpart; e.rpart = w.rpart; e.nh = w.nh; e.nseg = w.nseg;
  e.rm = a->running_mean; e.rv = a->running_var; e.nbt = a->num_batches_tracked;
  e.momentum = a->momentum; e.eps = a->eps;
  e.update = a->training && a->running_mean != nullptr && a->running_var != nullptr;
  e.w2 = a->w2;
  e.R = w.R; e.Y = w.Y; e.A = w.A; e.Z = w.Z; e.T = w.T; e.S = w.S; e.G = w.gm; e.dgb = w.dgb;
  return e;
}

static int eb_check(const bigcn_ebgcn_t* a, size_t workspace_bytes, const void* workspace, EbWs& w) {
  BIGCN_CHECK_ARG(a != nullptr && a->N >= 0 && a->B >= 0 && a->K > 0 && a->E >= 0, "ebgcn_conv2: bad dimensions");
  BIGCN_CHECK_ARG(a->N == 0 || (a->h1 && (a->x || a->x_ptr) && a->batch && a->w2),
                  "ebgcn_conv2: NULL h1, x (and x_ptr), batch or w2");
  BIGCN_CHECK_ARG(a->B == 0 || (a->rootindex && a->node_ptr), "ebgcn_conv2: NULL rootindex or node_ptr");
  BIGCN_CHECK_ARG(a->E == 0 || a->edge_index, "ebgcn_conv2: NULL edge_index");
  BIGCN_CHECK_ARG((a->bn_weight == nullptr) == (a->bn_bias == nullptr), "ebgcn_conv2: bn_weight and bn_bias go together");
  BIGCN_CHECK_ARG((a->running_mean == nullptr) == (a->running_var == nullptr),
                  "ebgcn_conv2: running_mean and running_var go together");
  BIGCN_CHECK_ARG(!(a->training && a->running_mean && a->momentum < 0.f && !a->num_batches_tracked),
                  "ebgcn_conv2: momentum=None needs num_batches_tracked");
  const bool csr = a->x == nullptr;
  w = carve_eb(a->N, a->B, a->K, a->E, csr, nullptr, 0);
  BIGCN_CHECK_ARG(workspace && workspace_bytes >= w.total, "ebgcn_conv2: workspace too small (%zu < %zu)", workspace_bytes,
                  w.total);
  w = carve_eb(a->N, a->B, a->K, a->E, csr, const_cast<void*>(workspace), workspace_bytes);
  return 0;
}

}  // namespace bigcn

using namespace bigcn;

extern "C" size_t bigcn_ebgcn_conv2_workspace_bytes(int64_t N, int64_t B, int64_t K, int64_t E) {
  return carve_eb(N, B, K, E, false, nullptr, 0).total;
}

extern "C" size_t bigcn_ebgcn_conv2_csr_workspace_bytes(int64_t N, int64_t B, int64_t K, int64_t E) {
  return carve_eb(N, B, K, E, true, nullptr, 0).total;
}

extern "C" int bigcn_ebgcn_conv2_forward(const bigcn_ebgcn_t* a, float* out, int32_t* flags, void* workspace,
                                         size_t workspace_bytes, bigcn_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  EbWs w;
  if (int rc = eb_check(a, workspace_bytes, workspace, w)) return rc;
  BIGCN_CHECK_ARG(flags && (a->N == 0 || out), "ebgcn_conv2_forward: NULL out or flags");
  const int64_t N = a->N, B = a->B, K = a->K, E = a->E;
  // the structure with the edge id as the sort payload, and the tree offsets of the batch vector
  const int64_t* eis[1] = {a->edge_index};
  const int64_t Es[1] = {E};
  int32_t* eids[2] = {w.G.in_eid, w.G.out_eid};
  if (int rc = graph_prep_impl(1, eis, Es, N, a->batch, B, a->deg_by, &w.G.g, a->node_ptr, flags, w.prep_ws, w.prep_bytes,
                               st, eids))
    return rc;
  if (N == 0) return 0;
  const float* ew = a->edge_weight;
  if (ew == nullptr) {
    if (int rc = wfeat_ones(w.ones, E, st)) return rc;
    ew = w.ones;
  }
  if (int rc = wfeat_prep(w.G, a->edge_index, E, ew, N, a->deg_by, w.in_w, w.out_w, flags, st)) return rc;
  if (B > 0) {
    k_eb_roots<<<(unsigned)ceil_div(B, 256), 256, 0, st>>>(a->rootindex, a->node_ptr, B, N, w.root, flags);
    BIGCN_CHECK_LAUNCH("k_eb_roots");
    if (a->x == nullptr) {
      k_eb_root_csr<<<(unsigned)B, 128, 0, st>>>(w.root, a->x_ptr, a->x_col, a->x_val, K, w.Xr, w.rmap, flags);
      BIGCN_CHECK_LAUNCH("k_eb_root_csr");
    }
  }
  Eb e = eb_args(a, w);
  const int mode = eb_mode(a);
  const unsigned cols = (unsigned)ceil_div(H + K, 256);
  if (mode == 0) {
    for (int pass = 0; pass < 2; ++pass) {
      if (pass == 0) k_eb_hstat<0><<<w.nh, 256, 0, st>>>(e);
      else k_eb_hstat<1><<<w.nh, 256, 0, st>>>(e);
      BIGCN_CHECK_LAUNCH("k_eb_hstat");
      if (B > 0) {
        const dim3 g((unsigned)ceil_div(K, 256), w.nseg);
        if (pass == 0) k_eb_rstat<0><<<g, 256, 0, st>>>(e);
        else k_eb_rstat<1><<<g, 256, 0, st>>>(e);
        BIGCN_CHECK_LAUNCH("k_eb_rstat");
      } else {
        cudaMemsetAsync(w.rpart, 0, (size_t)w.nseg * 2 * K * sizeof(double), st);
      }
      k_eb_stat_fin<<<cols, 256, 0, st>>>(e, pass);
      BIGCN_CHECK_LAUNCH("k_eb_stat_fin");
    }
  } else {
    k_eb_stat_fin<<<cols, 256, 0, st>>>(e, mode);
    BIGCN_CHECK_LAUNCH("k_eb_stat_fin");
  }
  if (B > 0) {
    k_eb_root_r<<<eb_grid(B * K, 256), 256, 0, st>>>(e);
    BIGCN_CHECK_LAUNCH("k_eb_root_r");
    const float* w2b[1] = {a->w2 + H};
    if (int rc = xw_dispatch(w.R, B, K, w2b, 1, H + K, w.wT, w.Y, H, BIGCN_GEMM_FP32, st)) return rc;
  }
  k_eb_mix<<<w.nh, 256, 0, st>>>(e);
  BIGCN_CHECK_LAUNCH("k_eb_mix");
  return w_propagate_launch(w.G.g.in_ptr, w.G.g.in_idx, w.G.in_eid, w.G.norm_e, w.G.norm_self, w.Z, a->b2, out, N, true,
                            st);
}

extern "C" int bigcn_ebgcn_conv2_backward(const bigcn_ebgcn_t* a, const float* out, const float* grad_out, float* dh1,
                                          float* d_bn_weight, float* d_bn_bias, float* dw2, float* db2,
                                          float* d_edge_weight, void* workspace, size_t workspace_bytes,
                                          bigcn_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  EbWs w;
  if (int rc = eb_check(a, workspace_bytes, workspace, w)) return rc;
  const int64_t N = a->N, B = a->B, K = a->K, E = a->E;
  BIGCN_CHECK_ARG(dw2 && db2 && (N == 0 || (out && grad_out && dh1)), "ebgcn_conv2_backward: NULL argument");
  if (N == 0) {
    cudaMemsetAsync(dw2, 0, (size_t)H * (H + K) * sizeof(float), st);
    cudaMemsetAsync(db2, 0, H * sizeof(float), st);
    if (d_bn_weight) cudaMemsetAsync(d_bn_weight, 0, (size_t)(H + K) * sizeof(float), st);
    if (d_bn_bias) cudaMemsetAsync(d_bn_bias, 0, (size_t)(H + K) * sizeof(float), st);
    if (d_edge_weight && E > 0) cudaMemsetAsync(d_edge_weight, 0, (size_t)E * sizeof(float), st);
    return 0;
  }
  Eb e = eb_args(a, w);
  const int mode = eb_mode(a);
  k_eb_gmask<<<eb_grid(N * H, 256), 256, 0, st>>>(grad_out, out, N * H, w.gm);
  BIGCN_CHECK_LAUNCH("k_eb_gmask");
  if (int rc = colsum64_launch(w.gm, N, w.cspart, db2, st)) return rc;
  // T = A-hat^T G: the by-source CSR with the same per-edge norms
  if (int rc = w_propagate_launch(w.G.g.out_ptr, w.G.g.out_idx, w.G.out_eid, w.G.norm_e, w.G.norm_self, w.gm, nullptr,
                                  w.T, N, false, st))
    return rc;
  if (d_edge_weight != nullptr) {
    if (int rc = w_edge_dot_launch(a->edge_index, E, N, w.gm, w.Z, w.a_e, w.a_self, st)) return rc;
    WGradArgs ga{};
    ga.d[0] = WGradDir{w.G, a->edge_index, E, a->edge_weight ? a->edge_weight : w.ones, w.a_e, w.a_self, w.ddeg,
                       d_edge_weight};
    ga.N = N;
    ga.deg_by_source = a->deg_by == BIGCN_DEG_BY_SOURCE;
    if (int rc = wfeat_edge_grad(ga, 1, st)) return rc;
  }
  // dW2a = T^T A
  OuterArgs oa{};
  oa.u[0] = w.T; oa.v[0] = w.A; oa.part[0] = w.opart; oa.N = N;
  OuterReduceArgs orr{};
  orr.part[0] = w.opart; orr.dst[0] = dw2; orr.ld = H + K; orr.nchunk = op_chunks(N);
  if (int rc = outer64_launch(oa, orr, 1, st)) return rc;
  // S per tree, dW2b = S^T R
  if (B > 0) {
    SegSumArgs sg{};
    sg.t[0] = w.T; sg.out[0] = w.S; sg.node_ptr = a->node_ptr;
    if (int rc = segsum_launch(sg, B, 1, st)) return rc;
  }
  if (int rc = dw_fp32(w.R, B, K, w.S, H, H, w.dwpart, dw2, H + K, H, nullptr, 0, 0, st)) return rc;
  // bn1: the root columns over trees, the h1 columns over rows
  if (mode != 3) {
    if (B > 0) {
      k_eb_root_bwd<<<dim3((unsigned)ceil_div(K, 128), w.nseg), 128, 0, st>>>(e);
      BIGCN_CHECK_LAUNCH("k_eb_root_bwd");
    } else {
      cudaMemsetAsync(w.rpart, 0, (size_t)w.nseg * 2 * K * sizeof(double), st);
    }
  }
  k_eb_hbwd1<<<w.nh, 256, 0, st>>>(e);
  BIGCN_CHECK_LAUNCH("k_eb_hbwd1");
  if (mode != 3) {
    k_eb_bwd_fin<<<(unsigned)ceil_div(H + K, 256), 256, 0, st>>>(e, d_bn_weight, d_bn_bias);
    BIGCN_CHECK_LAUNCH("k_eb_bwd_fin");
  }
  k_eb_hbwd2<<<eb_grid(N * H, 256), 256, 0, st>>>(e, mode, dh1);
  BIGCN_CHECK_LAUNCH("k_eb_hbwd2");
  return 0;
}
