// On-device batch assembly + DropEdge (SURVEY.md 8f, row N2): replaces, for a dataset kept
// resident in HBM, what BiGraphDataset.__getitem__ (Process/dataset.py:64-99) and PyG's
// Batch.from_data_list collate (model/Twitter/BiGCN_Twitter.py:168) do on the host per batch:
//   * DropEdge: keep int(e * (1 - rate)) positions of a tree's edge list, uniformly without
//     replacement, order preserved, drawn independently for the TD list and for the BU list
//     (dataset.py:68-90; random.sample -> the k smallest of per-position Philox keys);
//   * collate: concatenate x, offset edge_index / BU_edge_index / rootindex by the cumulative
//     node count, batch[i] = tree of node i, y.
// The packed dataset keeps x either as CSR (the `index:count` pairs getTwittergraph.py:16-24 reads,
// never densified), so the assembled batch feeds the BIGCN_GEMM_SPARSE path directly, or as dense
// fp32 / bf16 rows (PHEME's sentence embeddings), gathered by k_asm_dense_rows into a dense [n, K] x
// for the tensor-core modes.
// Offsets per tree are computed by the caller on the host from the (host-known) tree sizes:
// nothing here synchronises.
#include <algorithm>

#include "kernels.cuh"

namespace bigcn {

struct AsmArgs {
  // packed dataset
  const int64_t* node_ptr;   // [T+1]
  const int64_t* edge_ptr;   // [T+1]
  const int32_t* edge_src;   // [E_all] local ids: row 0 of the tree's edgeindex (parent)
  const int32_t* edge_dst;   // [E_all] row 1 (child)
  const int64_t* x_ptr;      // [N_all+1]
  const int32_t* x_col;
  const float* x_val;
  const int32_t* root_local; // [T]
  const int64_t* y_all;      // [T]
  // this batch
  const int64_t* tree_id;    // [B]
  const int64_t* node_off;   // [B+1]
  const int64_t* td_off;     // [B+1] kept TD edges
  const int64_t* bu_off;     // [B+1]
  const int64_t* nnz_off;    // [B+1]
  int64_t B, E_td, E_bu;
  uint32_t k0, k1;           // Philox key (seed)
  // outputs
  int64_t* edge_index;       // [2][E_td]
  int64_t* bu_edge_index;    // [2][E_bu]
  int64_t* batch;            // [N]
  int64_t* rootindex;        // [B]
  int64_t* y;                // [B]
  int32_t* ox_ptr;           // [N+1]
  int32_t* ox_col;
  float* ox_val;
  // edge weights (k_asm_edges<true> only), as bit patterns: copied, never converted
  const uint32_t* ew_all[2]; // [E_all] per tree edge: TD, BU
  uint32_t* ew[2];           // [E_td], [E_bu] per kept edge, aligned with edge_index / bu_edge_index
};

// nodes, features, labels: CTA per tree
__global__ void __launch_bounds__(256) k_asm_nodes(AsmArgs a) {
  const int64_t b = blockIdx.x;
  const int64_t t = a.tree_id[b];
  const int64_t n0 = a.node_ptr[t], n = a.node_ptr[t + 1] - n0;
  const int64_t off = a.node_off[b];
  if (a.x_ptr == nullptr) {   // dense features: k_asm_dense_rows copies the rows
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) a.batch[off + i] = b;
    if (threadIdx.x == 0) {
      a.rootindex[b] = off + a.root_local[t];
      a.y[b] = a.y_all[t];
    }
    return;
  }
  const int64_t z0 = a.x_ptr[n0], nz = a.x_ptr[n0 + n] - z0;
  const int64_t zoff = a.nnz_off[b];
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    a.batch[off + i] = b;
    a.ox_ptr[off + i] = (int32_t)(zoff + (a.x_ptr[n0 + i] - z0));
  }
  for (int64_t p = threadIdx.x; p < nz; p += blockDim.x) {
    a.ox_col[zoff + p] = a.x_col[z0 + p];
    a.ox_val[zoff + p] = a.x_val[z0 + p];
  }
  if (threadIdx.x == 0) {
    a.rootindex[b] = off + a.root_local[t];
    a.y[b] = a.y_all[t];
    if (b == a.B - 1) a.ox_ptr[off + n] = (int32_t)(zoff + nz);
  }
}

// edges.  DropEdge = a uniformly random k-subset of the e positions, order preserved
// (random.sample(range(e), k) followed by sorted(), dataset.py:72-75,84-87).
// CTA per (tree, direction): every position draws a 32-bit Philox key; a 32-step bisection finds
// the k-th smallest key v; positions with key < v are kept, plus the first ones with key == v
// until k are kept (ties, ~e^2 / 2^33 likely, resolved by position); an ordered block scan
// compacts the kept edges.  Every k-subset is equally likely (up to those ties).
// Weighted (W): the kept edge's weight goes to the same output position as the edge, in the same launch.
constexpr int DE_MAX = 8192;   // edges per tree handled in shared memory (32 KB of keys)

__device__ __forceinline__ uint32_t edge_key(const AsmArgs& a, int64_t t, int dir, int64_t i) {
  const Philox4 r = philox4x32_10((uint32_t)(i >> 2), (uint32_t)(t & 0xffffffffll), (uint32_t)((uint64_t)t >> 32),
                                  0x44450000u + (uint32_t)dir, a.k0, a.k1);
  return philox_elem(r, (int)(i & 3));
}

__device__ __forceinline__ int block_sum128(int v, int* red) {   // 128 threads, all get the total
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL_MASK, v, o);
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  return red[0] + red[1] + red[2] + red[3];
}

template <bool W>
__global__ void __launch_bounds__(128) k_asm_edges(AsmArgs a) {
  __shared__ uint32_t key[DE_MAX];
  __shared__ int red[4];
  __shared__ int wbase[4];
  const int64_t b = blockIdx.x >> 1;
  const int dir = (int)(blockIdx.x & 1);          // 0: TD list [row; col], 1: BU list [col; row]
  const int64_t t = a.tree_id[b];
  const int64_t e0 = a.edge_ptr[t];
  const int e = (int)(a.edge_ptr[t + 1] - e0);
  const int64_t* offs = dir ? a.bu_off : a.td_off;
  const int64_t o0 = offs[b];
  const int k = (int)(offs[b + 1] - o0);
  const int64_t noff = a.node_off[b];
  int64_t* out = dir ? a.bu_edge_index : a.edge_index;
  const int64_t E = dir ? a.E_bu : a.E_td;
  auto emit = [&](int i, int64_t pos) {
    const int64_t s = a.edge_src[e0 + i] + noff, d = a.edge_dst[e0 + i] + noff;
    out[o0 + pos] = dir ? d : s;
    out[E + o0 + pos] = dir ? s : d;
    if constexpr (W) a.ew[dir][o0 + pos] = a.ew_all[dir][e0 + i];
  };
  if (k >= e) {   // rate 0 (or nothing to drop): plain offset copy
    for (int i = threadIdx.x; i < e; i += 128) emit(i, i);
    return;
  }
  if (e > DE_MAX) {   // very large tree: Knuth's selection sampling (TAOCP 3.4.2 S) by one thread
    if (threadIdx.x == 0) {
      int kept = 0;
      for (int i = 0; i < e && kept < k; ++i) {
        const uint32_t u = edge_key(a, t, dir, i);
        // u / 2^32 < (k - kept) / (e - i)
        if ((unsigned long long)u * (unsigned long long)(e - i) < ((unsigned long long)(k - kept) << 32)) emit(i, kept++);
      }
    }
    return;
  }
  for (int i = threadIdx.x; i < e; i += 128) key[i] = edge_key(a, t, dir, i);
  __syncthreads();
  // smallest v with #{key <= v} >= k
  uint32_t lo = 0u, hi = 0xffffffffu;
  while (lo < hi) {
    const uint32_t mid = lo + ((hi - lo) >> 1);
    int c = 0;
    for (int i = threadIdx.x; i < e; i += 128) c += key[i] <= mid;
    if (block_sum128(c, red) >= k) hi = mid;
    else lo = mid + 1;
  }
  const uint32_t v = lo;
  int below = 0;
  for (int i = threadIdx.x; i < e; i += 128) below += key[i] < v;
  const int ties_kept = k - block_sum128(below, red);     // how many of the key == v positions are kept
  // ordered compaction, 128 positions per round
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int base = 0, ties_seen = 0;
  for (int i0 = 0; i0 < e; i0 += 128) {
    const int i = i0 + threadIdx.x;
    const bool in = i < e;
    const bool lt = in && key[i] < v, eq = in && key[i] == v;
    // position among the ties (block-ordered)
    const unsigned mq = __ballot_sync(FULL_MASK, eq);
    __syncthreads();
    if (lane == 0) wbase[w] = __popc(mq);
    __syncthreads();
    int tie_rank = ties_seen + __popc(mq & ((1u << lane) - 1u));
    for (int q = 0; q < w; ++q) tie_rank += wbase[q];
    const int ties_round = wbase[0] + wbase[1] + wbase[2] + wbase[3];
    const bool keep = lt || (eq && tie_rank < ties_kept);
    const unsigned mk = __ballot_sync(FULL_MASK, keep);
    __syncthreads();
    if (lane == 0) wbase[w] = __popc(mk);
    __syncthreads();
    int pos = base + __popc(mk & ((1u << lane) - 1u));
    for (int q = 0; q < w; ++q) pos += wbase[q];
    if (keep) emit(i, pos);
    base += wbase[0] + wbase[1] + wbase[2] + wbase[3];
    ties_seen += ties_round;
  }
}

// Dense feature rows.  Tree b's rows [node_ptr[tree_id[b]], +n_b) of x_all go to rows [node_off[b], +n_b) of ox,
// every row K * elem_bytes bytes; the batch's x is the concatenation of B byte ranges.
//   * Work split: the batch's units, in chunks of DR_THREADS * DR_UNROLL, are dealt out in contiguous runs to a grid
//     sized to the machine -- not a CTA per tree, since a PHEME batch mixes single-node trees with 300-node ones, and
//     one such tree is 118 MB in bf16 at K = 196,608.
//   * Offsets: tree_id / node_off usually sit in pinned host memory, a PCIe round trip per read.  Each CTA stages the
//     (source - destination) row delta of the trees its run touches into shared memory once, read by parallel threads;
//     a row's tree comes from the batch vector k_asm_nodes has just written to device memory.  No device scratch
//     array is needed, and no per-chunk search through host memory.  When node_off is pinned host memory, the host
//     reads the row count at launch: the grid is sized to the chunks (a 24-tree PHEME batch needs ~45 CTAs, not 4 per
//     SM, each of which would otherwise wait on the same PCIe read before it knows it has nothing to do).
//   * Units: 16 bytes (LDG.128 / STG.128) when the row bytes and both pointers allow it, else 4 or 2; integers
//     throughout, so every bit pattern (NaN payloads, -0.0) is copied as it is.  DR_UNROLL loads in flight per thread.
//   * Unit indices are 64-bit; the row / column split of a unit uses a 32-bit multiply-shift division by the row's
//     unit count on offsets below 2^31 (row_units < 2^30, so row remainder + chunk stays below that).
constexpr int DR_THREADS = 256, DR_UNROLL = 8, DR_TREES = 512;

struct DenseRowArgs {
  const int64_t* node_ptr;
  const int64_t* tree_id;
  const int64_t* node_off;
  const int64_t* batch;    // [N] tree of each batch row, written by k_asm_nodes
  const void* x;           // [N_all, K]
  void* ox;                // [N, K]
  int64_t B;
  int64_t n;               // rows of the batch (node_off[B]) when the host could read it, else -1
  uint32_t row_units;      // units per row
  uint32_t mul, shift;     // v / row_units == (umulhi(v, mul) + v) >> shift for every 32-bit v
};

__device__ __forceinline__ uint32_t dr_div(const DenseRowArgs& a, uint32_t v) {
  return (uint32_t)(((uint64_t)__umulhi(v, a.mul) + v) >> a.shift);
}

template <typename U>
__global__ void __launch_bounds__(DR_THREADS) k_asm_dense_rows(DenseRowArgs a) {
  __shared__ int64_t s_delta[DR_TREES];
  __shared__ int64_t s_n, s_row0, s_row1;
  const U* __restrict__ src = static_cast<const U*>(a.x);
  U* __restrict__ dst = static_cast<U*>(a.ox);
  const int64_t ru = a.row_units;
  if (threadIdx.x == 0) s_n = a.n >= 0 ? a.n : a.node_off[a.B];
  __syncthreads();
  constexpr int64_t CH = (int64_t)DR_THREADS * DR_UNROLL;
  const int64_t total = s_n * ru;
  const int64_t per = ((total + CH - 1) / CH + gridDim.x - 1) / gridDim.x;     // chunks per CTA
  const int64_t lo = min(total, (int64_t)blockIdx.x * per * CH), hi = min(total, lo + per * CH);
  if (lo >= hi) return;
  const int64_t b_lo = a.batch[lo / ru], b_hi = a.batch[(hi - 1) / ru] + 1;
  for (int64_t b0 = b_lo; b0 < b_hi; b0 += DR_TREES) {
    const int nb = (int)min((int64_t)DR_TREES, b_hi - b0);
    __syncthreads();   // the previous round is done with s_delta / s_row*
    for (int j = threadIdx.x; j < nb; j += DR_THREADS) {
      const int64_t off = a.node_off[b0 + j];
      s_delta[j] = a.node_ptr[a.tree_id[b0 + j]] - off;
      if (j == 0) s_row0 = off;
    }
    if (threadIdx.x == 0) s_row1 = a.node_off[b0 + nb];
    __syncthreads();
    const int64_t u0 = max(lo, s_row0 * ru), u1 = min(hi, s_row1 * ru);
    if (u0 >= u1) continue;
    int64_t row = u0 / ru;
    uint32_t rem = (uint32_t)(u0 - row * ru);      // unit u0 + c sits at (row, rem + c) with rem + c < 2^31
    for (int64_t u = u0; u < u1; u += CH) {
      U v[DR_UNROLL];
#pragma unroll
      for (int i = 0; i < DR_UNROLL; ++i) {
        const uint32_t c = (uint32_t)(i * DR_THREADS) + threadIdx.x;
        if (u + c < u1) {
          const uint32_t q = dr_div(a, rem + c);
          const int64_t r = row + q;
          const int64_t j = __ldg(a.batch + r) - b0;
          v[i] = __ldg(src + (r + s_delta[j]) * ru + (rem + c - q * a.row_units));
        }
      }
#pragma unroll
      for (int i = 0; i < DR_UNROLL; ++i) {
        const uint32_t c = (uint32_t)(i * DR_THREADS) + threadIdx.x;
        if (u + c < u1) dst[u + c] = v[i];
      }
      const uint32_t q = dr_div(a, rem + (uint32_t)CH);
      row += q;
      rem = rem + (uint32_t)CH - q * a.row_units;
    }
  }
}

}  // namespace bigcn

using namespace bigcn;

// weights (NULL = unweighted): checked, then laid into the assembly arguments
static int asm_weights(AsmArgs& a, const bigcn_asm_weights_t* w, const char* who) {
  if (w == nullptr) return 0;
  BIGCN_CHECK_ARG(w->td_weight && (a.E_td == 0 || w->edge_weight) && (a.E_bu == 0 || w->bu_edge_weight),
                  "%s: NULL weight array (td_weight, and an output for every non-empty direction)", who);
  a.ew_all[0] = reinterpret_cast<const uint32_t*>(w->td_weight);
  a.ew_all[1] = reinterpret_cast<const uint32_t*>(w->bu_weight ? w->bu_weight : w->td_weight);
  a.ew[0] = reinterpret_cast<uint32_t*>(w->edge_weight);
  a.ew[1] = reinterpret_cast<uint32_t*>(w->bu_edge_weight);
  return 0;
}
static void asm_edges_launch(const AsmArgs& a, bool weighted, cudaStream_t st) {
  if (weighted) k_asm_edges<true><<<(unsigned)(2 * a.B), 128, 0, st>>>(a);
  else k_asm_edges<false><<<(unsigned)(2 * a.B), 128, 0, st>>>(a);
}

static int assemble_csr(const int64_t* node_ptr, const int64_t* edge_ptr, const int32_t* edge_src,
                        const int32_t* edge_dst, const int64_t* x_ptr, const int32_t* x_col,
                        const float* x_val, const int32_t* root_local, const int64_t* y_all,
                        const int64_t* tree_id, const int64_t* node_off, const int64_t* td_off,
                        const int64_t* bu_off, const int64_t* nnz_off, int64_t B, int64_t E_td,
                        int64_t E_bu, uint64_t seed, int64_t* edge_index, int64_t* bu_edge_index,
                        int64_t* batch, int64_t* rootindex, int64_t* y, int32_t* ox_ptr, int32_t* ox_col,
                        float* ox_val, const bigcn_asm_weights_t* w, bigcn_stream_t stream) {
  BIGCN_CHECK_ARG(B >= 0 && E_td >= 0 && E_bu >= 0, "assemble_batch: bad sizes");
  if (B == 0) return 0;
  BIGCN_CHECK_ARG(node_ptr && edge_ptr && x_ptr && root_local && y_all && tree_id && node_off && td_off && bu_off &&
                      nnz_off && batch && rootindex && y && ox_ptr,
                  "assemble_batch: NULL argument");
  AsmArgs a{};
  a.node_ptr = node_ptr; a.edge_ptr = edge_ptr; a.edge_src = edge_src; a.edge_dst = edge_dst;
  a.x_ptr = x_ptr; a.x_col = x_col; a.x_val = x_val; a.root_local = root_local; a.y_all = y_all;
  a.tree_id = tree_id; a.node_off = node_off; a.td_off = td_off; a.bu_off = bu_off; a.nnz_off = nnz_off;
  a.B = B; a.E_td = E_td; a.E_bu = E_bu;
  a.k0 = (uint32_t)(seed & 0xffffffffull); a.k1 = (uint32_t)(seed >> 32);
  a.edge_index = edge_index; a.bu_edge_index = bu_edge_index; a.batch = batch; a.rootindex = rootindex; a.y = y;
  a.ox_ptr = ox_ptr; a.ox_col = ox_col; a.ox_val = ox_val;
  if (int rc = asm_weights(a, w, "assemble_batch")) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  k_asm_nodes<<<(unsigned)B, 256, 0, st>>>(a);
  BIGCN_CHECK_LAUNCH("k_asm_nodes");
  asm_edges_launch(a, w != nullptr, st);
  BIGCN_CHECK_LAUNCH("k_asm_edges");
  return 0;
}

static int assemble_dense(const int64_t* node_ptr, const int64_t* edge_ptr, const int32_t* edge_src,
                          const int32_t* edge_dst, const int32_t* root_local, const int64_t* y_all,
                          const int64_t* tree_id, const int64_t* node_off, const int64_t* td_off,
                          const int64_t* bu_off, int64_t B, int64_t E_td, int64_t E_bu, uint64_t seed,
                          int64_t* edge_index, int64_t* bu_edge_index, int64_t* batch,
                          int64_t* rootindex, int64_t* y, const void* x_all, int64_t K,
                          int32_t elem_bytes, void* ox, const bigcn_asm_weights_t* w, bigcn_stream_t stream) {
  BIGCN_CHECK_ARG(B >= 0 && E_td >= 0 && E_bu >= 0, "assemble_batch_dense: bad sizes");
  BIGCN_CHECK_ARG(elem_bytes == 2 || elem_bytes == 4,
                  "assemble_batch_dense: elem_bytes must be 2 (bf16) or 4 (fp32), got %d", (int)elem_bytes);
  BIGCN_CHECK_ARG(K >= 1 && K * elem_bytes < (1ll << 30),
                  "assemble_batch_dense: K = %lld (rows of 1 .. 2^30 - 1 bytes)", (long long)K);
  if (B == 0) return 0;
  BIGCN_CHECK_ARG(node_ptr && edge_ptr && root_local && y_all && tree_id && node_off && td_off && bu_off && batch &&
                      rootindex && y && x_all && ox,
                  "assemble_batch_dense: NULL argument");
  BIGCN_CHECK_ARG(((uintptr_t)x_all | (uintptr_t)ox) % (uintptr_t)elem_bytes == 0,
                  "assemble_batch_dense: x_all and ox must be aligned to elem_bytes (%d)", (int)elem_bytes);
  AsmArgs a{};
  a.node_ptr = node_ptr; a.edge_ptr = edge_ptr; a.edge_src = edge_src; a.edge_dst = edge_dst;
  a.root_local = root_local; a.y_all = y_all;
  a.tree_id = tree_id; a.node_off = node_off; a.td_off = td_off; a.bu_off = bu_off;
  a.B = B; a.E_td = E_td; a.E_bu = E_bu;
  a.k0 = (uint32_t)(seed & 0xffffffffull); a.k1 = (uint32_t)(seed >> 32);
  a.edge_index = edge_index; a.bu_edge_index = bu_edge_index; a.batch = batch; a.rootindex = rootindex; a.y = y;
  if (int rc = asm_weights(a, w, "assemble_batch_dense")) return rc;
  // the largest unit (16, 4 or 2 bytes) that divides the row bytes and both base addresses
  const uint64_t row_bytes = (uint64_t)K * (uint64_t)elem_bytes;
  const uint64_t align = row_bytes | (uint64_t)(uintptr_t)x_all | (uint64_t)(uintptr_t)ox;
  const int unit = align % 16 == 0 ? 16 : align % 4 == 0 ? 4 : 2;
  DenseRowArgs d{};
  d.node_ptr = node_ptr; d.tree_id = tree_id; d.node_off = node_off; d.batch = batch;
  d.x = x_all; d.ox = ox; d.B = B;
  d.row_units = (uint32_t)(row_bytes / unit);
  uint32_t l = 0;
  while ((1ull << l) < d.row_units) ++l;
  d.shift = l;
  d.mul = (uint32_t)((((1ull << l) - d.row_units) << 32) / d.row_units + 1);
  cudaStream_t st = (cudaStream_t)stream;
  k_asm_nodes<<<(unsigned)B, 256, 0, st>>>(a);
  BIGCN_CHECK_LAUNCH("k_asm_nodes");
  // the caller wrote node_off before this call; when it is pinned host memory its last entry is readable here
  d.n = -1;
  cudaPointerAttributes pa;
  if (cudaPointerGetAttributes(&pa, node_off) == cudaSuccess && pa.type == cudaMemoryTypeHost && pa.hostPointer)
    d.n = static_cast<const int64_t*>(pa.hostPointer)[B];
  else
    (void)cudaGetLastError();   // device memory, or a pointer CUDA does not know: the kernel reads node_off[B]
  int64_t grid64 = 4ll * num_sms();
  if (d.n >= 0) grid64 = std::min(grid64, (d.n * (int64_t)d.row_units + DR_THREADS * DR_UNROLL - 1) / (DR_THREADS * DR_UNROLL));
  const unsigned grid = (unsigned)grid64;
  if (grid > 0) {
    if (unit == 16) k_asm_dense_rows<uint4><<<grid, DR_THREADS, 0, st>>>(d);
    else if (unit == 4) k_asm_dense_rows<uint32_t><<<grid, DR_THREADS, 0, st>>>(d);
    else k_asm_dense_rows<uint16_t><<<grid, DR_THREADS, 0, st>>>(d);
    BIGCN_CHECK_LAUNCH("k_asm_dense_rows");
  }
  asm_edges_launch(a, w != nullptr, st);
  BIGCN_CHECK_LAUNCH("k_asm_edges");
  return 0;
}

extern "C" int bigcn_assemble_batch(const int64_t* node_ptr, const int64_t* edge_ptr, const int32_t* edge_src,
                                    const int32_t* edge_dst, const int64_t* x_ptr, const int32_t* x_col,
                                    const float* x_val, const int32_t* root_local, const int64_t* y_all,
                                    const int64_t* tree_id, const int64_t* node_off, const int64_t* td_off,
                                    const int64_t* bu_off, const int64_t* nnz_off, int64_t B, int64_t E_td,
                                    int64_t E_bu, uint64_t seed, int64_t* edge_index, int64_t* bu_edge_index,
                                    int64_t* batch, int64_t* rootindex, int64_t* y, int32_t* ox_ptr, int32_t* ox_col,
                                    float* ox_val, bigcn_stream_t stream) {
  return assemble_csr(node_ptr, edge_ptr, edge_src, edge_dst, x_ptr, x_col, x_val, root_local, y_all, tree_id, node_off,
                      td_off, bu_off, nnz_off, B, E_td, E_bu, seed, edge_index, bu_edge_index, batch, rootindex, y, ox_ptr,
                      ox_col, ox_val, nullptr, stream);
}

extern "C" int bigcn_assemble_batch_weighted(const int64_t* node_ptr, const int64_t* edge_ptr, const int32_t* edge_src,
                                             const int32_t* edge_dst, const int64_t* x_ptr, const int32_t* x_col,
                                             const float* x_val, const int32_t* root_local, const int64_t* y_all,
                                             const int64_t* tree_id, const int64_t* node_off, const int64_t* td_off,
                                             const int64_t* bu_off, const int64_t* nnz_off, int64_t B, int64_t E_td,
                                             int64_t E_bu, uint64_t seed, int64_t* edge_index, int64_t* bu_edge_index,
                                             int64_t* batch, int64_t* rootindex, int64_t* y, int32_t* ox_ptr,
                                             int32_t* ox_col, float* ox_val, const bigcn_asm_weights_t* weights,
                                             bigcn_stream_t stream) {
  BIGCN_CHECK_ARG(weights != nullptr, "assemble_batch_weighted: NULL weights (bigcn_assemble_batch takes none)");
  return assemble_csr(node_ptr, edge_ptr, edge_src, edge_dst, x_ptr, x_col, x_val, root_local, y_all, tree_id, node_off,
                      td_off, bu_off, nnz_off, B, E_td, E_bu, seed, edge_index, bu_edge_index, batch, rootindex, y, ox_ptr,
                      ox_col, ox_val, weights, stream);
}

extern "C" int bigcn_assemble_batch_dense(const int64_t* node_ptr, const int64_t* edge_ptr, const int32_t* edge_src,
                                          const int32_t* edge_dst, const int32_t* root_local, const int64_t* y_all,
                                          const int64_t* tree_id, const int64_t* node_off, const int64_t* td_off,
                                          const int64_t* bu_off, int64_t B, int64_t E_td, int64_t E_bu, uint64_t seed,
                                          int64_t* edge_index, int64_t* bu_edge_index, int64_t* batch,
                                          int64_t* rootindex, int64_t* y, const void* x_all, int64_t K,
                                          int32_t elem_bytes, void* ox, bigcn_stream_t stream) {
  return assemble_dense(node_ptr, edge_ptr, edge_src, edge_dst, root_local, y_all, tree_id, node_off, td_off, bu_off, B,
                        E_td, E_bu, seed, edge_index, bu_edge_index, batch, rootindex, y, x_all, K, elem_bytes, ox, nullptr,
                        stream);
}

extern "C" int bigcn_assemble_batch_dense_weighted(const int64_t* node_ptr, const int64_t* edge_ptr,
                                                   const int32_t* edge_src, const int32_t* edge_dst,
                                                   const int32_t* root_local, const int64_t* y_all,
                                                   const int64_t* tree_id, const int64_t* node_off,
                                                   const int64_t* td_off, const int64_t* bu_off, int64_t B, int64_t E_td,
                                                   int64_t E_bu, uint64_t seed, int64_t* edge_index,
                                                   int64_t* bu_edge_index, int64_t* batch, int64_t* rootindex,
                                                   int64_t* y, const void* x_all, int64_t K, int32_t elem_bytes,
                                                   void* ox, const bigcn_asm_weights_t* weights, bigcn_stream_t stream) {
  BIGCN_CHECK_ARG(weights != nullptr, "assemble_batch_dense_weighted: NULL weights (bigcn_assemble_batch_dense takes none)");
  return assemble_dense(node_ptr, edge_ptr, edge_src, edge_dst, root_local, y_all, tree_id, node_off, td_off, bu_off, B,
                        E_td, E_bu, seed, edge_index, bu_edge_index, batch, rootindex, y, x_all, K, elem_bytes, ox, weights,
                        stream);
}
