// Row-sparse view of X for conv1 (SURVEY.md 8f, row N1: the bag-of-words matrix the reference
// densifies at Process/getTwittergraph.py:16-24,67-72 is ~99.7 % zeros).
//
// gemm_mode = BIGCN_GEMM_SPARSE keeps the forward X*W as the exact-fp32 streaming scan over the
// dense X the caller hands over (xw.cu), but the scan also captures every row's non-zeros.
// From that capture this file builds, off the critical path (side stream):
//   CSR  (ptr[N+1], col, val, row)   exclusive scan of the row counts + compaction
//   CSC  (cptr[K+1], crow, cval)     stable LSD radix sort of the column keys (rows ascending
//                                    inside a column), hub-column list for the sweep
// and the weight gradient dW1 = T1^T X becomes a CSR sweep over the COLUMNS of X (gather.cuh):
//   dW1[o, k] = sum_{(i, v) in column k} v * T1[i, o]
// -- nnz * 128 FMAs instead of a second 600 MB pass over X.  Rows are added in ascending order
// with one fma chain per output, hot columns (a word present in most tweets) are split into
// fixed chunks combined in order: deterministic, no floating-point atomics.
// A caller that already has X in CSR form (sparse loader, host-side compaction of a dense
// host matrix) enters at the CSR stage and never materialises the dense matrix on the device.
#include "gather.cuh"

namespace bigcn {

constexpr int RSX_THREADS = 256;
constexpr int RSX_ROUNDS = 8;
constexpr int RSX_TILE = RSX_THREADS * RSX_ROUNDS;   // 2048 keys per block
constexpr int SCX_TILE = 2048;

int64_t xs_capacity(int64_t N, int64_t K) { return (N > 0 ? N : 1) * (K < XS_CAP_PER_ROW ? K : XS_CAP_PER_ROW); }
static int64_t xs_nblk(int64_t cap) { return ceil_div(cap > 0 ? cap : 1, RSX_TILE); }
static int64_t xs_nscan(int64_t N) { return ceil_div(N > 0 ? N : 1, SCX_TILE); }

XSparse xs_carve(Carver& c, int64_t N, int64_t K) {
  XSparse x{};
  x.N = N;
  x.K = K;
  x.cap = xs_capacity(N, K);
  x.state = c.take<int32_t>(4);
  x.cnt = c.take<int32_t>(N > 0 ? N : 1);
  x.ell_col = c.take<int32_t>((size_t)(N > 0 ? N : 1) * XS_ELL);
  x.ell_val = c.take<float>((size_t)(N > 0 ? N : 1) * XS_ELL);
  x.ptr = c.take<int32_t>(N + 1);
  x.col = c.take<int32_t>(x.cap);
  x.row = c.take<int32_t>(x.cap);
  x.val = c.take<float>(x.cap);
  x.keys[0] = c.take<int32_t>(x.cap);
  x.keys[1] = c.take<int32_t>(x.cap);
  x.perm[0] = c.take<int32_t>(x.cap);
  x.perm[1] = c.take<int32_t>(x.cap);
  x.hist = c.take<int32_t>((size_t)256 * xs_nblk(x.cap) + 4 * 256);   // + digit totals of up to four passes
  x.bsum = c.take<int32_t>(xs_nscan(N));
  x.cptr = c.take<int32_t>(K + 1);
  x.crow = c.take<int32_t>(x.cap);
  x.cval = c.take<float>(x.cap);
  for (int d = 0; d < 2; ++d) x.clong[d] = c.take<int32_t>(long_ws_ints(x.cap));
  return x;
}

// The same view for a caller's CSR (ptr / col / val are the caller's; no capture, so no row counts, ELL slots or scan
// partials): what k_xs_from_csr, the column sort and the column sweep touch, at the same capacity.
XSparse xs_carve_csr(Carver& c, int64_t N, int64_t K) {
  XSparse x{};
  x.N = N;
  x.K = K;
  x.cap = xs_capacity(N, K);
  x.state = c.take<int32_t>(4);
  x.row = c.take<int32_t>(x.cap);
  x.keys[0] = c.take<int32_t>(x.cap);
  x.keys[1] = c.take<int32_t>(x.cap);
  x.perm[0] = c.take<int32_t>(x.cap);
  x.perm[1] = c.take<int32_t>(x.cap);
  x.hist = c.take<int32_t>((size_t)256 * xs_nblk(x.cap) + 4 * 256);
  x.cptr = c.take<int32_t>(K + 1);
  x.crow = c.take<int32_t>(x.cap);
  x.cval = c.take<float>(x.cap);
  for (int d = 0; d < 2; ++d) x.clong[d] = c.take<int32_t>(long_ws_ints(x.cap));
  return x;
}

// ---- exclusive scan of the row counts -> ptr[N+1] -------------------------------------------
__device__ __forceinline__ int block_excl_scan256(int v, int* total) {
  __shared__ int warp_tot[8];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(FULL_MASK, inc, o);
    if (lane >= o) inc += t;
  }
  __syncthreads();
  if (lane == 31) warp_tot[w] = inc;
  __syncthreads();
  int pre = 0, tot = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int t = warp_tot[i];
    if (i < w) pre += t;
    tot += t;
  }
  *total = tot;
  return pre + inc - v;
}

__global__ void __launch_bounds__(256) k_xs_scan_blocksum(XSparse x) {
  if (blockIdx.x == 0 && threadIdx.x == 0) x.state[2] = 0;
  const int64_t base = (int64_t)blockIdx.x * SCX_TILE;
  int sum = 0;
#pragma unroll
  for (int it = 0; it < SCX_TILE / 256; ++it) {
    const int64_t i = base + it * 256 + threadIdx.x;
    if (i < x.N) sum += x.cnt[i];
  }
  int tot;
  block_excl_scan256(sum, &tot);
  if (threadIdx.x == 0) x.bsum[blockIdx.x] = tot;
}

__global__ void __launch_bounds__(256) k_xs_scan_apply(XSparse x) {
  int part = 0;
  for (int b = threadIdx.x; b < (int)blockIdx.x; b += 256) part += x.bsum[b];
  int block_prefix;
  block_excl_scan256(part, &block_prefix);
  constexpr int ITEMS = SCX_TILE / 256;
  const int64_t base = (int64_t)blockIdx.x * SCX_TILE + (int64_t)threadIdx.x * ITEMS;
  int v[ITEMS];
  int tsum = 0;
#pragma unroll
  for (int it = 0; it < ITEMS; ++it) {
    const int64_t i = base + it;
    v[it] = i < x.N ? x.cnt[i] : 0;
    tsum += v[it];
  }
  int tot;
  int run = block_prefix + block_excl_scan256(tsum, &tot);
#pragma unroll
  for (int it = 0; it < ITEMS; ++it) {
    const int64_t i = base + it;
    if (i < x.N) x.ptr[i] = run;
    run += v[it];
    if (i == x.N - 1) {
      x.ptr[x.N] = run;
      x.state[0] = run <= x.cap ? run : 0;   // nnz the later stages work on
      x.state[1] = run <= x.cap ? 0 : 1;     // more non-zeros than the sparse path is laid out for
      if (run > x.cap && x.flags) atomicOr(x.flags, BIGCN_FLAG_X_NOT_SPARSE);
    }
  }
  if (x.N == 0 && blockIdx.x == 0 && threadIdx.x == 0) {
    x.ptr[0] = 0;
    x.state[0] = 0;
    x.state[1] = 0;
  }
}

// ---- compaction: ELL capture (or, for rows with more than XS_ELL non-zeros, the dense row
// again) -> CSR (col, val, row) + sort keys / identity permutation --------------------------
__global__ void __launch_bounds__(256) k_xs_compact(XSparse x, const float* __restrict__ xd) {
  const int lane = threadIdx.x & 31;
  const int64_t w0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  // header of the hub-column list: counters and arrival flags start at zero
  {
    const int64_t hdr = long_hdr_ints(x.cap);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < hdr; i += (int64_t)gridDim.x * blockDim.x) {
      x.clong[0][i] = 0;
      x.clong[1][i] = 0;
    }
  }
  if (x.state[1]) return;
  for (int64_t i = w0; i < x.N; i += nw) {
    const int c = x.cnt[i];
    const int base = x.ptr[i];
    if (c <= XS_ELL) {
      for (int t = lane; t < c; t += 32) {
        const int k = x.ell_col[i * XS_ELL + t];
        x.col[base + t] = k;
        x.keys[0][base + t] = k;
        x.perm[0][base + t] = base + t;
        x.row[base + t] = (int32_t)i;
        x.val[base + t] = x.ell_val[i * XS_ELL + t];
      }
    } else {   // long row: ascending columns straight from the dense row
      int run = base;
      for (int64_t k0 = 0; k0 < x.K; k0 += 32) {
        const int64_t k = k0 + lane;
        const float v = k < x.K ? xd[i * x.K + k] : 0.f;
        const unsigned m = __ballot_sync(FULL_MASK, v != 0.f);
        if (v != 0.f) {
          const int p = run + __popc(m & ((1u << lane) - 1u));
          x.col[p] = (int32_t)k;
          x.keys[0][p] = (int32_t)k;
          x.perm[0][p] = p;
          x.row[p] = (int32_t)i;
          x.val[p] = v;
        }
        run += __popc(m);
      }
    }
  }
}

// caller-provided CSR (sparse input): keys / identity permutation / row ids
__global__ void __launch_bounds__(256) k_xs_from_csr(XSparse x) {
  const int lane = threadIdx.x & 31;
  const int64_t w0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  {
    const int64_t hdr = long_hdr_ints(x.cap);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < hdr; i += (int64_t)gridDim.x * blockDim.x) {
      x.clong[0][i] = 0;
      x.clong[1][i] = 0;
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    const int nnz = x.ptr[x.N];
    x.state[2] = 0;
    x.state[0] = nnz <= x.cap ? nnz : 0;
    x.state[1] = nnz <= x.cap ? 0 : 1;
    if (nnz > x.cap && x.flags) atomicOr(x.flags, BIGCN_FLAG_X_NOT_SPARSE);
  }
  if (x.ptr[x.N] > x.cap) return;
  for (int64_t i = w0; i < x.N; i += nw) {
    const int s = x.ptr[i], e = x.ptr[i + 1];
    for (int p = s + lane; p < e; p += 32) {
      int k = x.col[p];
      if (k < 0 || k >= x.K) {   // ignored by the forward product too (xw.cu)
        if (x.flags) atomicOr(x.flags, BIGCN_FLAG_X_CSR_RANGE);
        k = 0;
      }
      x.keys[0][p] = k;
      x.perm[0][p] = p;
      x.row[p] = (int32_t)i;
    }
  }
}

// ---- stable LSD radix sort of (column key, position), 8-bit digits ---------------------------
// digit totals of pass p live behind the per-block histograms (zeroed by xs_build_csc)
__device__ __forceinline__ int32_t* xs_dtot(const XSparse& x, int nblk, int pass) {
  return x.hist + (int64_t)256 * nblk + 256 * pass;
}

__global__ void __launch_bounds__(RSX_THREADS) k_xs_hist(XSparse x, int src, int shift, int nblk) {
  __shared__ int h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  const int n = x.state[0];
  const int64_t base = (int64_t)blockIdx.x * RSX_TILE;
  if (base < n) {
    const int32_t* keys = x.keys[src];
#pragma unroll
    for (int r = 0; r < RSX_ROUNDS; ++r) {
      const int64_t e = base + r * RSX_THREADS + threadIdx.x;
      if (e < n) atomicAdd(&h[(keys[e] >> shift) & 255], 1);
    }
  }
  __syncthreads();
  x.hist[(int64_t)threadIdx.x * nblk + blockIdx.x] = h[threadIdx.x];
  // integer atomics: the totals do not depend on the order of arrival
  if (base < n && h[threadIdx.x] != 0) atomicAdd(xs_dtot(x, nblk, shift >> 3) + threadIdx.x, h[threadIdx.x]);
}

// offsets of (digit, block) in digit-major order: 32 CTAs x 8 warps, warp = digit.  Every CTA scans the
// 256 digit totals (k_xs_hist summed them); each warp then scans its digit's per-block counts with
// coalesced loads.  Only the blocks that hold keys are walked.
__global__ void __launch_bounds__(256) k_xs_hscan(XSparse x, int nblk, int pass) {
  const int n = x.state[0];
  const int used = (int)min((int64_t)nblk, ((int64_t)n + RSX_TILE - 1) / RSX_TILE);
  __shared__ int s_base[256];
  int dummy;
  s_base[threadIdx.x] = block_excl_scan256(xs_dtot(x, nblk, pass)[threadIdx.x], &dummy);
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int d = blockIdx.x * 8 + (threadIdx.x >> 5);
  int32_t* row = x.hist + (int64_t)d * nblk;
  int run = s_base[d];
  for (int b0 = 0; b0 < used; b0 += 32) {
    const int b = b0 + lane;
    const int t = b < used ? row[b] : 0;
    int inc = t;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(FULL_MASK, inc, o);
      if (lane >= o) inc += u;
    }
    if (b < used) row[b] = run + inc - t;
    run += __shfl_sync(FULL_MASK, inc, 31);
  }
}

__global__ void __launch_bounds__(RSX_THREADS) k_xs_scatter(XSparse x, int src, int shift, int nblk) {
  const int n = x.state[0];
  const int64_t base = (int64_t)blockIdx.x * RSX_TILE;
  if (base >= n) return;
  const int32_t* keys = x.keys[src];
  const int32_t* vals = x.perm[src];
  int32_t* keys_o = x.keys[src ^ 1];
  int32_t* vals_o = x.perm[src ^ 1];
  __shared__ int dbase[256];
  __shared__ int wcnt[RSX_THREADS / 32][257];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  dbase[threadIdx.x] = x.hist[(int64_t)threadIdx.x * nblk + blockIdx.x];
  for (int r = 0; r < RSX_ROUNDS; ++r) {
    for (int i = threadIdx.x; i < (RSX_THREADS / 32) * 257; i += RSX_THREADS) (&wcnt[0][0])[i] = 0;
    __syncthreads();
    const int64_t e = base + r * RSX_THREADS + threadIdx.x;
    const bool valid = e < n;
    const int32_t key = valid ? keys[e] : 0;
    const int32_t val = valid ? vals[e] : 0;
    const int digit = valid ? ((key >> shift) & 255) : 256;
    const unsigned peers = __match_any_sync(FULL_MASK, digit);
    const int rank = __popc(peers & ((1u << lane) - 1u));
    if (rank == 0) wcnt[w][digit] = __popc(peers);
    __syncthreads();
    if (valid) {
      int pre = 0;
      for (int i = 0; i < w; ++i) pre += wcnt[i][digit];
      const int pos = dbase[digit] + pre + rank;
      keys_o[pos] = key;
      vals_o[pos] = val;
    }
    __syncthreads();
    int tot = 0;
#pragma unroll
    for (int i = 0; i < RSX_THREADS / 32; ++i) tot += wcnt[i][threadIdx.x];
    dbase[threadIdx.x] += tot;
    __syncthreads();
  }
}

// ---- CSC: gather (row, val) through the sorted permutation, column offsets from key changes ---
__global__ void __launch_bounds__(256) k_xs_finish(XSparse x, int src) {
  const int n = x.state[0];
  const int32_t* keys = x.keys[src];
  const int32_t* perm = x.perm[src];
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t0 == 0) x.state[2] = 1;   // the column-sorted copy of this batch exists
  if (n == 0) {
    for (int64_t k = t0; k <= x.K; k += stride) x.cptr[k] = 0;
    return;
  }
  for (int64_t q = t0; q < n; q += stride) {
    const int p = perm[q];
    x.crow[q] = x.row[p];
    const int kc = x.col[p];
    x.cval[q] = (kc >= 0 && kc < x.K) ? x.val[p] : 0.f;
    const int cur = keys[q];
    const int prev = q > 0 ? keys[q - 1] : -1;
    for (int k = prev + 1; k <= cur; ++k) x.cptr[k] = (int32_t)q;
    if (q == n - 1)
      for (int64_t k = cur + 1; k <= x.K; ++k) x.cptr[k] = n;
  }
}

// hub rows of a generic CSR (here: the columns of X)
__global__ void __launch_bounds__(256) k_long_build(const int32_t* __restrict__ ptr, int64_t nrows, int32_t* lng0,
                                                    int32_t* lng1, int64_t ecap) {
  const LongView L = long_view(blockIdx.y ? lng1 : lng0, ecap);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nrows; i += (int64_t)gridDim.x * blockDim.x) {
    const int len = ptr[i + 1] - ptr[i];
    if (len <= LONG_ROW) continue;
    int lch, nch;
    long_chunking(len, lch, nch);
    const int slot = atomicAdd(&L.cnt[0], 1);
    const int t0 = atomicAdd(&L.cnt[1], nch);
    L.row[slot] = (int32_t)i;
    L.item0[slot] = t0;
    for (int c = 0; c < nch; ++c) L.item_slot[t0 + c] = slot;
  }
}

static int radix_passes_for(int64_t K) {
  int bits = 1;
  while (((int64_t)1 << bits) < K) ++bits;
  return (bits + 7) / 8;
}

// row capture (or a caller's CSR) -> CSR (col, val, row) + sort keys / identity permutation
int xs_build_csr(const XSparse& x, const float* x_dense, bool from_capture, cudaStream_t st) {
  int grid_rows = (int)ceil_div(x.N > 0 ? x.N : 1, 8);
  const int cap_ctas = num_sms() * 4;
  if (grid_rows > cap_ctas) grid_rows = cap_ctas;
  if (from_capture) {
    const int nsb = (int)xs_nscan(x.N);
    k_xs_scan_blocksum<<<nsb, 256, 0, st>>>(x);
    BIGCN_CHECK_LAUNCH("k_xs_scan_blocksum");
    k_xs_scan_apply<<<nsb, 256, 0, st>>>(x);
    BIGCN_CHECK_LAUNCH("k_xs_scan_apply");
    k_xs_compact<<<grid_rows, 256, 0, st>>>(x, x_dense);
    BIGCN_CHECK_LAUNCH("k_xs_compact");
  } else {
    k_xs_from_csr<<<grid_rows, 256, 0, st>>>(x);
    BIGCN_CHECK_LAUNCH("k_xs_from_csr");
  }
  return 0;
}

// CSR -> column-sorted CSC (stable LSD radix sort of the column keys) + hub-column lists
int xs_sort_csc(const XSparse& x, cudaStream_t st) {
  const int nblk = (int)xs_nblk(x.cap);
  const int passes = radix_passes_for(x.K);
  cudaMemsetAsync(x.hist + (int64_t)256 * nblk, 0, 4 * 256 * sizeof(int32_t), st);   // digit totals
  int grid_keys = nblk;   // blocks past the live keys return at once
  for (int p = 0; p < passes; ++p) {
    k_xs_hist<<<grid_keys, RSX_THREADS, 0, st>>>(x, p & 1, 8 * p, nblk);
    BIGCN_CHECK_LAUNCH("k_xs_hist");
    k_xs_hscan<<<32, 256, 0, st>>>(x, nblk, p);
    BIGCN_CHECK_LAUNCH("k_xs_hscan");
    k_xs_scatter<<<grid_keys, RSX_THREADS, 0, st>>>(x, p & 1, 8 * p, nblk);
    BIGCN_CHECK_LAUNCH("k_xs_scatter");
  }
  const int cap_ctas = num_sms() * 4;
  int gf = (int)ceil_div(x.cap, 256);
  if (gf > cap_ctas) gf = cap_ctas;
  k_xs_finish<<<gf, 256, 0, st>>>(x, passes & 1);
  BIGCN_CHECK_LAUNCH("k_xs_finish");
  int gl = (int)ceil_div(x.K, 256);
  k_long_build<<<dim3(gl, 2), 256, 0, st>>>(x.cptr, x.K, x.clong[0], x.clong[1], x.cap);
  BIGCN_CHECK_LAUNCH("k_long_build");
  return 0;
}

// everything between the row capture / a caller's CSR and the column-sorted copy
int xs_build_csc(const XSparse& x, const float* x_dense, bool from_capture, cudaStream_t st) {
  if (int rc = xs_build_csr(x, x_dense, from_capture, st)) return rc;
  return xs_sort_csc(x, st);
}

// ---- dW1[o, k] = sum_{(i,v) in column k} v * T[i, o]: CSR sweep over the columns ------------
struct PostDw {
  static constexpr bool kPairs = false;
  static constexpr bool kInline = true;
  float* dw;          // [64][ldw] rows of this direction's lin.weight gradient
  int64_t ldw;
  const int32_t* state;
  __device__ __forceinline__ void operator()(int k, const float4& v, int sub, unsigned, float*) const {
    // a batch denser than the sparse layout allows must not pass for a gradient
    const bool bad = state[1] != 0 || state[2] == 0;
    const float nan = __int_as_float(0x7fc00000);
    float* p = dw + (int64_t)(4 * sub) * ldw + k;
    p[0] = bad ? nan : v.x;
    p[ldw] = bad ? nan : v.y;
    p[2 * ldw] = bad ? nan : v.z;
    p[3 * ldw] = bad ? nan : v.w;
  }
};

// 2 columns per half-warp block (a short column still holds up to LONG_ROW entries), 16 T rows
// staged per round: 72 KB per CTA, 3 CTAs per SM
constexpr int DW_R = 2, DW_Q = 16;

struct DwSweepArgs {
  XSparse x;
  const float* t;     // [N][ldt], direction d in columns [64 d, 64 d + 64)
  int64_t ldt;
  float* dw[2];
  int64_t ldw;
  int32_t cb;
};

template <int R, int Q, int MINB>
__global__ void __launch_bounds__(256, MINB) k_dw_sweep(DwSweepArgs a) {
  extern __shared__ __align__(128) float sweep_smem[];
  const int d = blockIdx.y;
  csr_sweep<R, Q, false>(Csr{a.x.cptr, a.x.crow, a.x.clong[d], a.x.cap}, WtVal{a.x.cval}, (int)a.x.K, a.cb, sweep_smem,
                         ValRow{a.t + d * H, a.ldt}, PostDw{a.dw[d], a.ldw, a.x.state});
}

template <int R, int Q, int MINB>
static int dw_sweep_launch(DwSweepArgs& a, int n_out, cudaStream_t st) {
  constexpr int smem = SweepSmem<R, Q>::kBytes;
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(k_dw_sweep<R, Q, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    attr = true;
  }
  // the work is in the hub columns (a bag-of-words matrix is Zipf-skewed: most non-zeros sit in
  // columns with more than LONG_ROW entries), i.e. in the (column, chunk) items every half-warp of
  // the grid picks up after the short columns: fill the machine whatever K is
  const int max_ctas = num_sms() * MINB;
  a.cb = 8;
  int grid = sweep_grid(a.x.K, R, a.cb, max_ctas);
  const int64_t by_items = ceil_div(a.x.cap / LONG_ROW, 16);
  if (grid < max_ctas) grid = (int)(by_items < max_ctas ? (by_items > grid ? by_items : grid) : max_ctas);
  k_dw_sweep<R, Q, MINB><<<dim3(grid, n_out / H), 256, smem, st>>>(a);
  BIGCN_CHECK_LAUNCH("k_dw_sweep");
  return 0;
}

int dw_sparse(const XSparse& x, const float* t, int64_t ldt, int n_out, float* dw_a, float* dw_b, int64_t ldw,
              cudaStream_t st) {
  if (x.K == 0) return 0;
  DwSweepArgs a{};
  a.x = x; a.t = t; a.ldt = ldt; a.dw[0] = dw_a; a.dw[1] = dw_b; a.ldw = ldw;
  return dw_sweep_launch<DW_R, DW_Q, 3>(a, n_out, st);
}

}  // namespace bigcn
