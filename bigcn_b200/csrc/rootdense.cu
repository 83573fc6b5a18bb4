// The root half of conv2.lin in TRAINING mode when the root features are DENSE (PHEME: 768-d sentence embeddings, about
// half of them positive after the relu).
//
// Reference: x = dropout(relu(cat(h1, root_extend)))  ->  conv2.lin   (BiGCN_Twitter.py:45-56, BU :95-105); the lin of
// the concatenation splits into a1 W2a^T (the mix kernel) and, for node i of tree b,
//     R[i, :] = sum_k keep(i, 64 + k) * relu(x[root_b, k]) * W2b^T[k, :]          (z += scale * R)
// and the matching weight gradient  dW2b[o, k] = scale * sum_i keep(i, 64 + k) * relu(x[root_b(i), k]) * T2[i, o].
//
// With bag-of-words roots (~20 non-zero columns) both walk the tree's short column list inside the mix kernel and the
// (part, reduce) pair of propagate.cu.  With dense roots that list is the whole row: the per-node loop in the mix
// kernel becomes a serial chain of K / 16 rounds (68 us for a 240-node batch, and the whole step 12x an inference pass
// at 4096 trees), and the column-per-CTA fallback of the gradient re-reads a T2 row for every kept (node, column)
// pair.  These two kernels are the same sums as register-tiled products whose [node, column] operand is synthesised in
// shared memory from the root row and one Philox block per four columns -- every T2 / W2b element is read once per
// tile, not once per pair.  Summation order of R: columns ascending, one fma chain per output -- the order of the list
// walk (a dropped or zero term adds an exact zero), so with one column split R is bit-identical to it; small batches
// split the columns over several CTAs (a CTA's K / 32 chunks are one latency chain) and the mix kernel adds the
// partials in split order.  dW2b: node segments, nodes ascending inside a segment, segments combined in order.
// Everything is deterministic; no atomics.
#include "kernels.cuh"
#include "gather.cuh"

namespace bigcn {

constexpr int RD_KC = 32;   // columns per chunk

// relu(x[root, k .. k + 3]) masked by the dropout decisions of node `node` for columns 64 + k .. 64 + k + 3 (k % 4 == 0:
// exactly one Philox block, the block the list walk of the mix kernel draws for these columns).  T = float, or
// __nv_bfloat16 when x is bf16 (BIGCN_GEMM_BF16: widened exactly, so the same values as from the fp32 copy)
template <typename T>
__device__ __forceinline__ void masked_root_quad(const float* __restrict__ x, int64_t root_row, int64_t K, int64_t k,
                                                 const DropSpec& ds, int64_t node, float out[4]) {
  out[0] = out[1] = out[2] = out[3] = 0.f;
  if (root_row < 0 || k >= K) return;
  const T* xr = reinterpret_cast<const T*>(x) + root_row * K + k;
  float v[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) v[j] = k + j < K ? fmaxf(x_f32(__ldg(xr + j)), 0.f) : 0.f;
  if ((v[0] > 0.f) | (v[1] > 0.f) | (v[2] > 0.f) | (v[3] > 0.f)) {
    const Philox4 r = drop_block(ds, node, (uint32_t)((H + k) >> 2));
    out[0] = r.x >= ds.thresh ? v[0] : 0.f;
    out[1] = r.y >= ds.thresh ? v[1] : 0.f;
    out[2] = r.z >= ds.thresh ? v[2] : 0.f;
    out[3] = r.w >= ds.thresh ? v[3] : 0.f;
  }
}

// ---- forward: R[i, 0:64] for 32 * NPT nodes per CTA ----------------------------------------------
// 256 threads; thread t owns outputs 4 q .. + 3 and 32 + 4 q .. + 3 (q = t & 7: the eight lanes of a quarter-warp read
// 128 contiguous bytes of a W row, conflict-free) of the NPT consecutive nodes NPT * (t >> 3) ...  The operand tile is
// stored [column][node], so a thread's nodes come as one vector load that its quarter-warp shares.  Shared-memory
// wavefronts per column and warp: NPT = 2: 2 + 8 for 8 packed fmas per thread; NPT = 4: 4 + 8 for 16 (the first
// version -- outputs 8 q .. + 7, a two-way bank conflict on every W load -- ran at 44 % conflicted wavefronts and was
// bound by them: profiles/r02e_prof_rootdense_*).
template <int NPT, typename T>
__global__ void __launch_bounds__(256) k_root_dense(RootDenseArgs a) {
  constexpr int TN = 32 * NPT;
  __shared__ __align__(16) float sW[RD_KC][H];
  __shared__ __align__(16) float sA[RD_KC][TN + 4];
  __shared__ int64_t sRoot[TN];
  const int d = blockIdx.y, split = blockIdx.z;
  // this CTA's column range: whole chunks, split evenly
  const int64_t nchunk = (a.K + RD_KC - 1) / RD_KC;
  const int64_t kbeg = nchunk * split / a.ksplit * RD_KC, kend = min(a.K, nchunk * (split + 1) / a.ksplit * RD_KC);
  const int64_t i0 = (int64_t)blockIdx.x * TN;
  const int t = threadIdx.x, oq = t & 7, n0 = NPT * (t >> 3);
  const DropSpec ds = a.drop[d];
  if (t < TN) sRoot[t] = i0 + t < a.N ? a.rootindex[a.batch[i0 + t]] : -1;
  float4 acc[NPT][2];
#pragma unroll
  for (int r = 0; r < NPT; ++r) acc[r][0] = acc[r][1] = make_float4(0.f, 0.f, 0.f, 0.f);
  __syncthreads();
  for (int64_t k0 = kbeg; k0 < kend; k0 += RD_KC) {
#pragma unroll
    for (int u = 0; u < 2; ++u) {   // the W2b^T chunk: 32 x 64 floats
      const int f = (t + 256 * u) * 4, kk = f >> 6, o = f & 63;
      const float4 w = k0 + kk < kend ? ld4(a.w2bT[d] + (k0 + kk) * H + o) : make_float4(0.f, 0.f, 0.f, 0.f);
      st4(&sW[kk][o], w);
    }
#pragma unroll
    for (int u = 0; u < NPT; ++u) {   // the masked root operand: TN nodes x 8 quads, consecutive lanes = consecutive nodes
      const int q = t + 256 * u, node = q % TN, kq = q / TN;
      float m[4];
      masked_root_quad<T>(a.x, sRoot[node], a.K, k0 + 4 * kq, ds, a.node_id_base + i0 + node, m);
#pragma unroll
      for (int j = 0; j < 4; ++j) sA[4 * kq + j][node] = k0 + 4 * kq + j < kend ? m[j] : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int kk = 0; kk < RD_KC; ++kk) {
      float av[NPT];
      if constexpr (NPT == 4) {
        const float4 v = ld4(&sA[kk][n0]);
        av[0] = v.x; av[1] = v.y; av[2] = v.z; av[3] = v.w;
      } else {
        const float2 v = *reinterpret_cast<const float2*>(&sA[kk][n0]);
        av[0] = v.x; av[1] = v.y;
      }
      const float4 w0 = ld4(&sW[kk][4 * oq]), w1 = ld4(&sW[kk][32 + 4 * oq]);
#pragma unroll
      for (int r = 0; r < NPT; ++r) {
        fma4(acc[r][0], av[r], w0);
        fma4(acc[r][1], av[r], w1);
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int r = 0; r < NPT; ++r) {
    const int64_t i = i0 + n0 + r;
    if (i < a.N) {
      float* out = a.r[d] + ((int64_t)split * a.N + i) * H;
      st4(out + 4 * oq, acc[r][0]);
      st4(out + 32 + 4 * oq, acc[r][1]);
    }
  }
}

// column splits: enough CTAs for the machine on small batches, within the partial buffer (RD_CAP_ROWS rows per direction)
int root_dense_splits(int64_t N, int64_t K) {
  if (N <= 0) return 1;
  int64_t s = RD_CAP_ROWS / N;
  const int64_t nchunk = ceil_div(K, (int64_t)RD_KC);
  if (s > 8) s = 8;
  if (s > nchunk) s = nchunk;
  return (int)(s < 1 ? 1 : s);
}

int root_dense_forward(const RootDenseArgs& a, int ndir, cudaStream_t st) {
  if (a.N == 0) return 0;
  const dim3 g4((unsigned)ceil_div(a.N, 128), ndir, a.ksplit), g2((unsigned)ceil_div(a.N, 64), ndir, a.ksplit);
  if (a.N * ndir * a.ksplit >= (int64_t)128 * 2 * num_sms()) {   // enough 128-node tiles for two waves: the leaner inner loop
    if (a.x_bf16) k_root_dense<4, __nv_bfloat16><<<g4, 256, 0, st>>>(a);
    else k_root_dense<4, float><<<g4, 256, 0, st>>>(a);
  } else {
    if (a.x_bf16) k_root_dense<2, __nv_bfloat16><<<g2, 256, 0, st>>>(a);
    else k_root_dense<2, float><<<g2, 256, 0, st>>>(a);
  }
  BIGCN_CHECK_LAUNCH("k_root_dense");
  return 0;
}

// ---- backward: dW2b partials, CTA = 128 columns x one node segment -------------------------------
// thread t owns outputs 4 q .. + 3 and 32 + 4 q .. + 3 (q = t & 7) of the four columns k0 + 4 (t >> 3) .. + 3; nodes of
// the segment in tiles of 32, ascending.  The operand tile is stored [node][column]: a thread's four columns are one
// vector load.  Per node and warp: 4 + 8 shared-memory wavefronts for 16 packed fmas per thread.
constexpr int RD_BK = 128;   // columns per CTA
template <typename T>
__global__ void __launch_bounds__(256) k_dw2b_dense_part(Dw2bDenseArgs a) {
  __shared__ __align__(16) float sT[32][H];
  __shared__ __align__(16) float sA[32][RD_BK + 4];
  const int d = blockIdx.z, seg = blockIdx.y;
  const int64_t k0 = (int64_t)blockIdx.x * RD_BK;
  const int t = threadIdx.x, oq = t & 7, kq = t >> 3;   // columns k0 + 4 kq .. + 3
  const DropSpec ds = a.drop[d];
  const int64_t s0 = (int64_t)seg * a.seg_rows, s1 = min(a.N, s0 + a.seg_rows);
  float4 acc[4][2];
#pragma unroll
  for (int c = 0; c < 4; ++c) acc[c][0] = acc[c][1] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int64_t i0 = s0; i0 < s1; i0 += 32) {
#pragma unroll
    for (int u = 0; u < 2; ++u) {   // T2 rows of the tile
      const int f = (t + 256 * u) * 4, nn = f >> 6, o = f & 63;
      const float4 v = i0 + nn < s1 ? ld4(a.t2[d] + (i0 + nn) * H + o) : make_float4(0.f, 0.f, 0.f, 0.f);
      st4(&sT[nn][o], v);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {   // the masked root operand: 32 nodes x 32 quads, consecutive lanes = consecutive quads
      const int q = t + 256 * u, node = q >> 5, cq = q & 31;
      const int64_t i = i0 + node;
      float m[4];
      masked_root_quad<T>(a.x, i < s1 ? a.rootindex[a.batch[i]] : -1, a.K, k0 + 4 * cq, ds, a.node_id_base + i, m);
      st4(&sA[node][4 * cq], make_float4(m[0], m[1], m[2], m[3]));
    }
    __syncthreads();
#pragma unroll 4
    for (int nn = 0; nn < 32; ++nn) {
      const float4 av = ld4(&sA[nn][4 * kq]);
      const float4 t0 = ld4(&sT[nn][4 * oq]), t1 = ld4(&sT[nn][32 + 4 * oq]);
      fma4(acc[0][0], av.x, t0); fma4(acc[0][1], av.x, t1);
      fma4(acc[1][0], av.y, t0); fma4(acc[1][1], av.y, t1);
      fma4(acc[2][0], av.z, t0); fma4(acc[2][1], av.z, t1);
      fma4(acc[3][0], av.w, t0); fma4(acc[3][1], av.w, t1);
    }
    __syncthreads();
  }
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const int64_t k = k0 + 4 * kq + c;
    if (k < a.K) {
      float* p = a.part[d] + ((int64_t)seg * a.K + k) * H;
      st4(p + 4 * oq, acc[c][0]);
      st4(p + 32 + 4 * oq, acc[c][1]);
    }
  }
}

// dW2[o][64 + k] = scale * (part[0][k][o] + part[1][k][o] + ...), segments ascending
__global__ void __launch_bounds__(256) k_dw2b_dense_reduce(Dw2bDenseArgs a) {
  const int d = blockIdx.y;
  const int64_t idx = (int64_t)blockIdx.x * 256 + threadIdx.x;   // k * 64 + o
  if (idx >= a.K * H) return;
  float s = 0.f;
  for (int seg = 0; seg < a.nseg; ++seg) s += a.part[d][(int64_t)seg * a.K * H + idx];
  const int64_t k = idx >> 6, o = idx & 63;
  a.dw2[d][o * a.ld + H + k] = s * a.drop[d].scale;
}

int dw2b_dense_segments(int64_t N, int64_t B, int64_t K) {
  // the partials live in the S buffer of the sparse-root path: (dw2b_blocks(N) + B) * DW2B_CAP * 64 floats per direction,
  // never less than one segment (carve_features)
  int64_t fit = ((int64_t)dw2b_blocks(N) + B) * DW2B_CAP / (K > 0 ? K : 1);
  int64_t want = ceil_div(N > 0 ? N : 1, 512);
  if (want > 64) want = 64;
  if (want > fit) want = fit;
  return (int)(want < 1 ? 1 : want);
}

int dw2b_dense_backward(const Dw2bDenseArgs& a0, int ndir, cudaStream_t st) {
  if (a0.K == 0) return 0;
  Dw2bDenseArgs a = a0;
  a.seg_rows = ceil_div(ceil_div(a.N > 0 ? a.N : 1, a.nseg), 32) * 32;
  const dim3 grid((unsigned)ceil_div(a.K, RD_BK), a.nseg, ndir);
  if (a.x_bf16) k_dw2b_dense_part<__nv_bfloat16><<<grid, 256, 0, st>>>(a);
  else k_dw2b_dense_part<float><<<grid, 256, 0, st>>>(a);
  BIGCN_CHECK_LAUNCH("k_dw2b_dense_part");
  k_dw2b_dense_reduce<<<dim3((unsigned)ceil_div(a.K * H, 256), ndir), 256, 0, st>>>(a);
  BIGCN_CHECK_LAUNCH("k_dw2b_dense_reduce");
  return 0;
}

}  // namespace bigcn
