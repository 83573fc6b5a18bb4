// Propagate, conv2 input mix, readout and their backward kernels.
//
// Replaces, per direction (BiGCN_Twitter.py:26-67 / 77-114):
//   MessagePassing.propagate + bias [torch_geometric]        -> k_propagate / k_prop1_mix
//   root-extend loops, cat, relu, dropout (:45-54)             -> k_root_nz, k_root_proj, k_prop1_mix
//   conv2.lin on the [h1 | root_extend] tensor (:56)           -> k_prop1_mix (never materialises N x 5064)
//   second root-extend + scatter_mean (:58-65)                 -> k_readout
// All kernels are warp-per-row over 64-wide fp32 rows (float2 per lane, 256 B coalesced),
// gather through the int32 CSR built by graph_prep, sum in COO' order with separate
// multiply and add (bit-identical to the CPU index_add_ order), and use no atomics.
#include "gather.cuh"

namespace bigcn {

// ---------------------------------------------------------------- A-hat / A-hat^T propagate
// out = A-hat h (+ bias)(relu): the CSR sweep of gather.cuh with a bias / relu / store epilogue.
constexpr int PROP_R = 8, PROP_Q = 8;     // 64 KB stage per CTA, 3 CTAs per SM
constexpr int MIX_R = 2, MIX_Q = 4;       // 24 KB stage + 16 KB W2a per CTA, 4 CTAs per SM (64 registers): the
                                          // heavy per-row epilogue wants warps in flight more than a deep stage

struct PostBiasRelu {
  static constexpr bool kPairs = false;
  static constexpr bool kInline = true;
  const float* bias;
  float* out;
  int64_t ldo;
  int relu;
  float4 b;
  __device__ __forceinline__ void operator()(int i, float4 v, int sub, unsigned, float*) const {
    if (bias) {
      v.x = __fadd_rn(v.x, b.x);
      v.y = __fadd_rn(v.y, b.y);
      v.z = __fadd_rn(v.z, b.z);
      v.w = __fadd_rn(v.w, b.w);
    }
    if (relu) {
      v.x = fmaxf(v.x, 0.f);
      v.y = fmaxf(v.y, 0.f);
      v.z = fmaxf(v.z, 0.f);
      v.w = fmaxf(v.w, 0.f);
    }
    st4(out + (int64_t)i * ldo + 4 * sub, v);
  }
};

template <class Wt>
__device__ __forceinline__ void propagate_dir(const PropArgs& a, const PropDir& p, const Wt& wt, float* sweep_smem) {
  const int sub = threadIdx.x & 15;
  PostBiasRelu post{p.bias, p.out, p.ldo, a.relu, make_float4(0.f, 0.f, 0.f, 0.f)};
  if (p.bias) post.b = ld4(p.bias + 4 * sub);
  csr_sweep<PROP_R, PROP_Q, true>(Csr{p.ptr, p.idx, p.lng, p.E}, wt, (int)a.N, a.cb, sweep_smem, ValRow{p.h, p.ldh}, post);
}
__global__ void __launch_bounds__(256, 3) k_propagate(PropArgs a) {
  extern __shared__ __align__(128) float sweep_smem[];
  const PropDir p = a.d[blockIdx.y];
  propagate_dir(a, p, WtGcn{p.dis}, sweep_smem);
}
// edge-weighted batch: p.dis holds the normalised self-loop weights, ew.w[d] the normalised weight of every entry of
// the CSR being swept (EntryW, weighted.cu)
__global__ void __launch_bounds__(256, 3) k_propagate_w(PropArgs a, EntryW ew) {
  extern __shared__ __align__(128) float sweep_smem[];
  const PropDir p = a.d[blockIdx.y];
  propagate_dir(a, p, WtEntry{ew.w[blockIdx.y], p.dis}, sweep_smem);
}

template <class K>
static void sweep_attr(K kernel, int smem) {
  cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
}

int propagate_launch(const PropArgs& a0, int ndir, cudaStream_t st, const EntryW* ew) {
  if (a0.N == 0) return 0;
  constexpr int smem = SweepSmem<PROP_R, PROP_Q>::kBytes;
  static bool attr = false;
  if (!attr) {
    sweep_attr(k_propagate, smem);
    sweep_attr(k_propagate_w, smem);
    attr = true;
  }
  PropArgs a = a0;
  const int max_ctas = num_sms() * 3;
  a.cb = sweep_cb(a.N, PROP_R, max_ctas);
  const dim3 grid(sweep_grid(a.N, PROP_R, a.cb, max_ctas), ndir);
  if (ew) {
    k_propagate_w<<<grid, 256, smem, st>>>(a, *ew);
    BIGCN_CHECK_LAUNCH("k_propagate_w");
    return 0;
  }
  k_propagate<<<grid, 256, smem, st>>>(a);
  BIGCN_CHECK_LAUNCH("k_propagate");
  return 0;
}

// ---------------------------------------------------------------- root non-zeros
// Per tree: the columns k with relu(x[root,k]) > 0, ascending, and their values.
// (root_extend of BiGCN_Twitter.py:45-50 is x1[rootindex[batch]]: only these columns
// can contribute to conv2 after the relu of :53.)
// CTA per tree: 8 warps ballot 32-column strips, a strip-count scan orders them, a second
// pass writes (col, val) at its rank and slot[k][b] = rank for the positive columns (column-major map,
// preset to -1, that the dW2b reduce uses to find a column's slot in each tree with coalesced loads).
// T = float, or __nv_bfloat16 when x is bf16 (BIGCN_GEMM_BF16: the values are widened exactly).
template <typename T>
__global__ void __launch_bounds__(256) k_root_nz(RootNzArgs a) {
  extern __shared__ int strip[];  // [nstrips] counts -> exclusive offsets
  __shared__ int s_total;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t b = blockIdx.x;
  const int nstrips = (int)((a.K + 31) / 32);
  const int64_t r = a.rootindex[b];
  const bool ok = r >= 0 && r < a.N;
  if (!ok && threadIdx.x == 0) atomicOr(a.flags, BIGCN_FLAG_ROOT_RANGE);
  const T* xr = reinterpret_cast<const T*>(a.x) + (ok ? r : 0) * a.K;
  for (int s = w; s < nstrips; s += 8) {
    const int64_t k = (int64_t)s * 32 + lane;
    const float v = (ok && k < a.K) ? x_f32(xr[k]) : 0.f;
    const unsigned m = __ballot_sync(FULL_MASK, v > 0.f);
    if (lane == 0) strip[s] = __popc(m);
  }
  __syncthreads();
  if (w == 0) {  // exclusive scan of the strip counts: contiguous chunk per lane
    const int per = (nstrips + 31) / 32;
    const int lo = min(lane * per, nstrips), hi = min(lo + per, nstrips);
    int sum = 0;
    for (int s = lo; s < hi; ++s) sum += strip[s];
    int inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(FULL_MASK, inc, o);
      if (lane >= o) inc += t;
    }
    int run = inc - sum;
    for (int s = lo; s < hi; ++s) {
      const int t = strip[s];
      strip[s] = run;
      run += t;
    }
    if (lane == 31) s_total = inc;
  }
  __syncthreads();
  for (int s = w; s < nstrips; s += 8) {
    const int64_t k = (int64_t)s * 32 + lane;
    const float v = (ok && k < a.K) ? x_f32(xr[k]) : 0.f;
    const unsigned m = __ballot_sync(FULL_MASK, v > 0.f);
    const int pos = strip[s] + __popc(m & ((1u << lane) - 1u));
    if (v > 0.f) {
      a.col[b * a.K + pos] = (int32_t)k;
      a.val[b * a.K + pos] = v;
      a.overflow[1 + k] = 1;   // column k is positive in some root row (same value from every writer)
      a.slot[k * a.B + b] = pos;  // column-major slot map, -1 (memset) everywhere else
    }
  }
  if (threadIdx.x == 0) {
    a.cnt[b] = s_total;
    if (s_total > a.cap) atomicOr(a.overflow, 1);
  }
}

// the same from a CSR of x (sparse input): the root row's positive entries in CSR order
__global__ void __launch_bounds__(256) k_root_nz_csr(RootNzArgs a, const int32_t* __restrict__ xptr,
                                                     const int32_t* __restrict__ xcol, const float* __restrict__ xval) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t b = blockIdx.x;
  if (w != 0) return;
  const int64_t r = a.rootindex[b];
  const bool ok = r >= 0 && r < a.N;
  if (!ok && lane == 0) atomicOr(a.flags, BIGCN_FLAG_ROOT_RANGE);
  const int s = ok ? xptr[r] : 0, e = ok ? xptr[r + 1] : 0;
  int n = 0;
  for (int p0 = s; p0 < e; p0 += 32) {
    const int p = p0 + lane;
    int k = 0;
    float v = 0.f;
    if (p < e) {
      k = xcol[p];
      v = xval[p];
    }
    const bool pos_ok = v > 0.f && k >= 0 && k < a.K;
    const unsigned m = __ballot_sync(FULL_MASK, pos_ok);
    if (pos_ok) {
      const int pos = n + __popc(m & ((1u << lane) - 1u));
      a.col[b * a.K + pos] = k;
      a.val[b * a.K + pos] = v;
      a.slot[(int64_t)k * a.B + b] = pos;
      a.overflow[1 + k] = 1;
    }
    n += __popc(m);
  }
  if (lane == 0) {
    a.cnt[b] = n;
    if (n > a.cap) atomicOr(a.overflow, 1);
  }
}

// eval mode: P[d][b][:] = relu(x_root[b]) * W2b_d^T, once per tree (SURVEY appendix A)
__global__ void __launch_bounds__(256) k_root_proj(RootProjArgs a) {
  const int d = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (b >= a.B) return;
  const int n = a.cnt[b];
  float2 acc = make_float2(0.f, 0.f);
  for (int t0 = 0; t0 < n; t0 += 32) {
    const int t = t0 + lane;
    int k = 0;
    float v = 0.f;
    if (t < n) {
      k = a.col[b * a.K + t];
      v = a.val[b * a.K + t];
    }
    const int m = min(32, n - t0);
    for (int l = 0; l < m; ++l) {
      const int kk = __shfl_sync(FULL_MASK, k, l);
      const float vv = __shfl_sync(FULL_MASK, v, l);
      const float2 w = *reinterpret_cast<const float2*>(a.w2bT[d] + (int64_t)kk * H + 2 * lane);
      acc.x = fmaf(vv, w.x, acc.x);
      acc.y = fmaf(vv, w.y, acc.y);
    }
  }
  *reinterpret_cast<float2*>(a.P[d] + b * H + 2 * lane) = acc;
}

// ---------------------------------------------------------------- conv1 propagate + conv2 input
// Per node i and direction d:
//   h1 = A-hat (XW1)[i] + b1                      (:42)    -> H1 (pre-relu, kept for :44 and backward)
//   a1 = dropout(relu(h1))                        (:53-54) -> A1 (kept for dW2a)
//   z  = a1 W2a^T + dropout(relu(x_root[b_i])) W2b^T   (:51-56, the lin of conv2 on the cat)
// The root part touches only the non-zero root columns (k_root_nz); one Philox block per
// lane decides which of them survive for this node.  Half-warp per row (float4 per lane):
// a lane's four columns are exactly one Philox block.
__device__ __forceinline__ void drop_quad(const DropSpec& ds, int64_t node, int sub, float4& a) {
  const Philox4 r = drop_block(ds, node, (uint32_t)sub);
  a.x = r.x >= ds.thresh ? __fmul_rn(a.x, ds.scale) : 0.f;
  a.y = r.y >= ds.thresh ? __fmul_rn(a.y, ds.scale) : 0.f;
  a.z = r.z >= ds.thresh ? __fmul_rn(a.z, ds.scale) : 0.f;
  a.w = r.w >= ds.thresh ? __fmul_rn(a.w, ds.scale) : 0.f;
}
// z[4*sub..] = sum_k av[k] * sW[k][4*sub..]: the half-warp parks av in shared memory and every
// lane reads it back as broadcast float4s (no shuffles), k ascending, one fma chain per output
__device__ __forceinline__ float4 matvec_smem(const float4& av, const float* __restrict__ sW, float* scratch,
                                              int sub, unsigned hm) {
  st4(scratch + 4 * sub, av);
  __syncwarp(hm);
  float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
  for (int k4 = 0; k4 < H / 4; ++k4) {
    const float4 a4 = ld4(scratch + 4 * k4);
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const float s = comp4(a4, c);
      const float4 w = ld4(sW + (4 * k4 + c) * H + 4 * sub);
      fma4(z, s, w);
    }
  }
  __syncwarp(hm);
  return z;
}

// two rows at once: every W row fetched from shared memory feeds both (half the LDS traffic, eight
// independent fma chains); per row the same k-ascending chain as matvec_smem
__device__ __forceinline__ void matvec2_smem(const float4& a0, const float4& a1, const float* __restrict__ sW,
                                             float* scratch, int sub, unsigned hm, float4& z0, float4& z1) {
  st4(scratch + 4 * sub, a0);
  st4(scratch + H + 4 * sub, a1);
  __syncwarp(hm);
  z0 = make_float4(0.f, 0.f, 0.f, 0.f);
  z1 = z0;
#pragma unroll 4
  for (int k4 = 0; k4 < H / 4; ++k4) {
    const float4 p4 = ld4(scratch + 4 * k4), q4 = ld4(scratch + H + 4 * k4);
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const float s0 = comp4(p4, c), s1 = comp4(q4, c);
      const float4 w = ld4(sW + (4 * k4 + c) * H + 4 * sub);
      fma4(z0, s0, w);
      fma4(z1, s1, w);
    }
  }
  __syncwarp(hm);
}

struct PostMix {
  static constexpr bool kPairs = true;
  static constexpr bool kInline = false;
  MixDir p;
  const float* sW;
  const int64_t* batch;
  const int32_t* rnz_cnt;
  const int32_t* rnz_col;
  const float* rnz_val;
  int64_t K, node_id_base;
  float4 b1;
  int root_splits;
  const float* root_r;
  int64_t root_stride;
  // bias, H1, relu, dropout, A1 of one row -> the conv2.lin input of its 64 hidden columns
  __device__ __forceinline__ float4 activate(int i, float4 h1, int sub) const {
    h1.x = __fadd_rn(h1.x, b1.x);
    h1.y = __fadd_rn(h1.y, b1.y);
    h1.z = __fadd_rn(h1.z, b1.z);
    h1.w = __fadd_rn(h1.w, b1.w);
    st4(p.h1 + (int64_t)i * H + 4 * sub, h1);
    float4 av = make_float4(fmaxf(h1.x, 0.f), fmaxf(h1.y, 0.f), fmaxf(h1.z, 0.f), fmaxf(h1.w, 0.f));
    if (p.drop.on) drop_quad(p.drop, node_id_base + i, sub, av);
    st4(p.a1 + (int64_t)i * H + 4 * sub, av);
    return av;
  }
  // root part of conv2.lin and the store of z
  __device__ __forceinline__ void finish(int i, float4 z, int sub, unsigned hm, float* scratch) const {
    const int64_t node = node_id_base + i;
    const int64_t b = batch[i];
    if (p.drop.on && root_splits > 0) {   // dense roots: k_root_dense left R[i] (one split: the sums of the walk below, in its order)
      float4 rv = ld4(root_r + (int64_t)i * H + 4 * sub);
      for (int s = 1; s < root_splits; ++s) {
        const float4 t = ld4(root_r + s * root_stride + (int64_t)i * H + 4 * sub);
        rv.x += t.x;
        rv.y += t.y;
        rv.z += t.z;
        rv.w += t.w;
      }
      z.x = fmaf(p.drop.scale, rv.x, z.x);
      z.y = fmaf(p.drop.scale, rv.y, z.y);
      z.z = fmaf(p.drop.scale, rv.z, z.z);
      z.w = fmaf(p.drop.scale, rv.w, z.w);
    } else if (p.drop.on) {
      const int n = rnz_cnt[b];
      float4 racc = make_float4(0.f, 0.f, 0.f, 0.f);
      unsigned long long kept = 0ull;   // bit t = root slot t survived for this node (slots 0..63)
      for (int t0 = 0; t0 < n; t0 += 16) {
        const int t = t0 + sub;
        int k = 0;
        float v = 0.f;
        bool keep = false;
        if (t < n) {
          k = rnz_col[b * K + t];
          v = rnz_val[b * K + t];
          const uint32_t c = (uint32_t)(H + k);
          const Philox4 r = drop_block(p.drop, node, c >> 2);
          keep = philox_elem(r, c & 3) >= p.drop.thresh;
        }
        // kept entries in ascending order: (k, v) pairs go through the scratch row
        unsigned mine = (__ballot_sync(hm, keep) >> (hm == 0xffffu ? 0 : 16)) & 0xffffu;
        if (t0 < 64) kept |= (unsigned long long)mine << t0;
        if (keep) {
          const int pos = __popc(mine & ((1u << sub) - 1u));
          reinterpret_cast<int*>(scratch)[pos] = k;
          scratch[16 + pos] = v;
        }
        __syncwarp(hm);
        const int cnt = __popc(mine);
        for (int q0 = 0; q0 < cnt; q0 += 4) {   // four W2b rows (L2) in flight, added in kept order
          float4 w[4];
          float vv[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            vv[u] = 0.f;
            w[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (q0 + u < cnt) {
              const int kk = reinterpret_cast<const int*>(scratch)[q0 + u];
              vv[u] = scratch[16 + q0 + u];
              w[u] = ld4(p.w2bT + (int64_t)kk * H + 4 * sub);
            }
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            if (q0 + u < cnt) fma4(racc, vv[u], w[u]);
          }
        }
        __syncwarp(hm);
      }
      // the backward's dW2b sums T2 rows over exactly these (node, slot) pairs: hand it the decisions
      if (sub == 0 && p.keep != nullptr) p.keep[i] = kept;
      z.x = fmaf(p.drop.scale, racc.x, z.x);
      z.y = fmaf(p.drop.scale, racc.y, z.y);
      z.z = fmaf(p.drop.scale, racc.z, z.z);
      z.w = fmaf(p.drop.scale, racc.w, z.w);
    } else {
      const float4 pv = ld4(p.P + b * H + 4 * sub);
      z.x += pv.x;
      z.y += pv.y;
      z.z += pv.z;
      z.w += pv.w;
    }
    st4(p.z + (int64_t)i * H + 4 * sub, z);
  }
  __device__ __forceinline__ void operator()(int i, float4 h1, int sub, unsigned hm, float* scratch) const {
    const float4 av = activate(i, h1, sub);
    finish(i, matvec_smem(av, sW, scratch, sub, hm), sub, hm, scratch);
  }
  // rows i (ok0) and i + 1 (ok1); scratch holds two rows
  __device__ __forceinline__ void pair(int i, float4 v0, bool ok0, float4 v1, bool ok1, int sub, unsigned hm,
                                       float* scratch) const {
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 a0 = ok0 ? activate(i, v0, sub) : zero;
    const float4 a1 = ok1 ? activate(i + 1, v1, sub) : zero;
    float4 z0, z1;
    matvec2_smem(a0, a1, sW, scratch, sub, hm, z0, z1);
    if (ok0) finish(i, z0, sub, hm, scratch);
    if (ok1) finish(i + 1, z1, sub, hm, scratch);
  }
};

template <int R, int Q, class Wt>
__device__ __forceinline__ void prop1_mix_dir(const MixArgs& a, const MixDir& p, const Wt& wt, float* sweep_smem,
                                              float* sW) {
  for (int i = threadIdx.x; i < H * H; i += blockDim.x) sW[i] = p.w2aT[i];
  // csr_sweep starts with a __syncthreads()
  const int sub = threadIdx.x & 15;
  PostMix post{p, sW, a.batch, a.rnz_cnt, a.rnz_col, a.rnz_val, a.K, a.node_id_base, ld4(p.b1 + 4 * sub), a.root_splits,
               a.root_r[blockIdx.y], a.N * H};
  csr_sweep<R, Q, true>(Csr{p.ptr, p.idx, p.lng, p.E}, wt, (int)a.N, a.cb, sweep_smem, ValRow{p.xw, a.ldxw}, post);
}
template <int R, int Q, int MINB>
__global__ void __launch_bounds__(256, MINB) k_prop1_mix(MixArgs a) {
  extern __shared__ __align__(128) float sweep_smem[];
  __shared__ __align__(16) float sW[H * H];
  const MixDir p = a.d[blockIdx.y];
  prop1_mix_dir<R, Q>(a, p, WtGcn{p.dis}, sweep_smem, sW);
}
// edge-weighted batch (see k_propagate_w): p.dis holds the self-loop weights
__global__ void __launch_bounds__(256, 4) k_prop1_mix_w(MixArgs a, EntryW ew) {
  extern __shared__ __align__(128) float sweep_smem[];
  __shared__ __align__(16) float sW[H * H];
  const MixDir p = a.d[blockIdx.y];
  prop1_mix_dir<MIX_R, MIX_Q>(a, p, WtEntry{ew.w[blockIdx.y], p.dis}, sweep_smem, sW);
}


// ---------------------------------------------------------------- readout
// feat[b, base_d + f]      = mean_{i in tree b} H2_d[i, f]           (scatter_mean, :65)
// feat[b, base_d + 64 + f] = H1_d[rootindex[b], f]                   (:58-63; the mean of n_b
//                            identical rows, taken as the row itself)
// Two launches, both with grids that depend on N and B only (no host sync on tree sizes):
//  part : one CTA per (tree, slice of RO_SLICE global rows) pair.  Trees are contiguous and
//         sorted, so the pair (slice g, tree b) has the unique id g + b; CTA x finds its tree by
//         bisecting f(b) = node_ptr[b] / RO_SLICE + b.  A 59k-node Weibo tree is spread over 116
//         CTAs, a batch of 10-node PHEME trees costs one small CTA per tree.  16 row lanes x
//         16 float4 lanes, 8 rows in flight per thread, fixed-order combine.
//  final: per tree, the slice partials in slice order, the divide, the positive counts the
//         backward uses for db2, and the root row of H1.
__global__ void __launch_bounds__(256) k_readout_part(ReadoutArgs a) {
  __shared__ __align__(16) float part[16][H];
  __shared__ __align__(16) float cpos[16][H];
  const int d = blockIdx.y;
  const int64_t x = blockIdx.x;
  int lo = 0, hi = (int)a.B - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if ((int64_t)(a.node_ptr[mid] / RO_SLICE) + mid <= x) lo = mid;
    else hi = mid - 1;
  }
  const int b = lo;
  const int64_t g = x - b;
  const int s = a.node_ptr[b], e = a.node_ptr[b + 1];
  const int64_t r0 = max((int64_t)s, g * RO_SLICE), r1 = min((int64_t)e, (g + 1) * RO_SLICE);
  if (r0 >= r1) return;   // not a (tree, slice) pair: never read by the final pass
  const int rl = threadIdx.x >> 4, sub = threadIdx.x & 15;
  const float* h2 = a.h2[d] + 4 * sub;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f), np = acc;
  for (int64_t i = r0 + rl; i < r1; i += 16 * 8) {
    float4 v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int64_t r = i + 16 * u;
      v[u] = r < r1 ? ld4(h2 + r * H) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w;
      np.x += v[u].x > 0.f ? 1.f : 0.f;
      np.y += v[u].y > 0.f ? 1.f : 0.f;
      np.z += v[u].z > 0.f ? 1.f : 0.f;
      np.w += v[u].w > 0.f ? 1.f : 0.f;
    }
  }
  st4(&part[rl][4 * sub], acc);
  st4(&cpos[rl][4 * sub], np);
  __syncthreads();
  if (threadIdx.x < 2 * H) {
    const int f = threadIdx.x & 63;
    const float(*src)[H] = threadIdx.x < H ? part : cpos;
    float t = 0.f;
#pragma unroll
    for (int r = 0; r < 16; ++r) t += src[r][f];
    a.scratch[(((int64_t)d * a.nitems + x) * 2 + (threadIdx.x >> 6)) * H + f] = t;
  }
}

__global__ void __launch_bounds__(256) k_readout_final(ReadoutArgs a) {
  const int64_t b = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 6);
  const int f = threadIdx.x & 63;
  if (b >= a.B) return;
  float mean[2], root[2], cnt[2];
  readout_final_tree(a, b, f, mean, root, cnt);
}

// scatter_mean backward on its own (the fused training path forms this inside k_propagate_g2):
// dh2[i][f] = grad_feat[batch[i]][f] / n_b.  Half-warp per row.
__global__ void __launch_bounds__(256) k_readout_bwd(const float* __restrict__ gfeat, int64_t ldg,
                                                     const int32_t* __restrict__ node_ptr, const int64_t* __restrict__ batch,
                                                     int64_t N, int64_t B, float* __restrict__ dh2) {
  const int sub = threadIdx.x & 15;
  for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 4; i < N; i += ((int64_t)gridDim.x * blockDim.x) >> 4) {
    const int64_t b = batch[i];
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
    if (b >= 0 && b < B) {
      const int n = node_ptr[b + 1] - node_ptr[b];
      const float inv_n = (float)(n > 0 ? n : 1);
      const float4 v = ld4(gfeat + b * ldg + 4 * sub);
      g = make_float4(__fdiv_rn(v.x, inv_n), __fdiv_rn(v.y, inv_n), __fdiv_rn(v.z, inv_n), __fdiv_rn(v.w, inv_n));
    }
    st4(dh2 + i * H + 4 * sub, g);
  }
}
int readout_bwd_launch(const float* gfeat, int64_t ldg, const int32_t* node_ptr, const int64_t* batch, int64_t N, int64_t B,
                       float* dh2, cudaStream_t st) {
  if (N == 0) return 0;
  int64_t g = ceil_div(N, 16);
  const int64_t cap = (int64_t)num_sms() * 8;
  if (g > cap) g = cap;
  k_readout_bwd<<<(int)g, 256, 0, st>>>(gfeat, ldg, node_ptr, batch, N, B, dh2);
  BIGCN_CHECK_LAUNCH("k_readout_bwd");
  return 0;
}

// ---------------------------------------------------------------- backward pieces
// Per tree: gs[d][b][f] = grad_feat[b][base_d + f] / n_b (scatter_mean backward), and the
// partial column sums of db2 = sum_i G2[i] = sum_b gs[b] * #{i in b : H2[i] > 0} using the
// positive counts the readout kept.  G2 itself is never materialised: k_propagate_g2 forms
// it on the fly while gathering.
__global__ void __launch_bounds__(256) k_gscale(GScaleArgs a) {
  __shared__ float red[4][H];
  const int d = blockIdx.y;
  const int g = threadIdx.x >> 6, f = threadIdx.x & 63;
  const int64_t base = (int64_t)blockIdx.x * GS_TREES;
  const int64_t end = min(a.B, base + GS_TREES);
  float acc = 0.f;
  for (int64_t b = base + g; b < end; b += 4) {
    const int n = a.node_ptr[b + 1] - a.node_ptr[b];
    const float gv = __fdiv_rn(a.grad_feat[b * 4 * H + a.feat_base[d] + f], (float)(n > 0 ? n : 1));
    a.gs[d][b * H + f] = gv;
    acc = fmaf(gv, a.pos[d][b * H + f], acc);
  }
  red[g][f] = acc;
  __syncthreads();
  if (g == 0) a.part[d][(int64_t)blockIdx.x * H + f] = ((red[0][f] + red[1][f]) + red[2][f]) + red[3][f];
}

// T2[j] = sum_{x in out(j)} (dis[j]*dis[x]) * G2[x] + dis[j]^2 * G2[j],
// G2[x] = [H2[x] > 0] * gs[batch[x]]   (relu and scatter_mean backward fused into the gather)
struct ValG2 {   // val(x) = [H2[x] > 0] * gs[batch[x]]
  static constexpr bool kHasAux = true;
  const float* h2;
  const float* gs;
  const int64_t* batch;
  __device__ __forceinline__ void fetch(float* dst, int j, int sub) const {
    cp_async_row16(dst + 4 * sub, h2 + (int64_t)j * H + 4 * sub);
  }
  __device__ __forceinline__ int aux(int j) const { return (int)batch[j]; }
  __device__ __forceinline__ float4 value(const float* slot, int b, int sub) const {
    const float4 hv = ld4(slot + 4 * sub);
    const float4 gv = ld4(gs + (int64_t)b * H + 4 * sub);
    return make_float4(hv.x > 0.f ? gv.x : 0.f, hv.y > 0.f ? gv.y : 0.f, hv.z > 0.f ? gv.z : 0.f,
                       hv.w > 0.f ? gv.w : 0.f);
  }
};
struct PostStore {
  static constexpr bool kPairs = false;
  static constexpr bool kInline = true;
  float* out;
  __device__ __forceinline__ void operator()(int i, const float4& v, int sub, unsigned, float*) const {
    st4(out + (int64_t)i * H + 4 * sub, v);
  }
};
template <class Wt>
__device__ __forceinline__ void propagate_g2_dir(const PropG2Args& a, const PropG2Dir& p, const Wt& wt, float* sweep_smem) {
  csr_sweep<PROP_R, PROP_Q, false>(Csr{p.ptr, p.idx, p.lng, p.E}, wt, (int)a.N, a.cb, sweep_smem,
                                   ValG2{p.h2, p.gs, a.batch}, PostStore{p.out});
}
__global__ void __launch_bounds__(256, 3) k_propagate_g2(PropG2Args a) {
  extern __shared__ __align__(128) float sweep_smem[];
  const PropG2Dir p = a.d[blockIdx.y];
  propagate_g2_dir(a, p, WtGcn{p.dis}, sweep_smem);
}
// edge-weighted batch (see k_propagate_w): by-source CSR, its own per-entry weights
__global__ void __launch_bounds__(256, 3) k_propagate_g2_w(PropG2Args a, EntryW ew) {
  extern __shared__ __align__(128) float sweep_smem[];
  const PropG2Dir p = a.d[blockIdx.y];
  propagate_g2_dir(a, p, WtEntry{ew.w[blockIdx.y], p.dis}, sweep_smem);
}

// out[f] = sum_chunk part[chunk][f]: 4 strided groups, fixed-order combine
__global__ void __launch_bounds__(256) k_colsum_reduce(ColsumArgs a) {
  __shared__ float red[4][H];
  const int j = blockIdx.x;
  const int g = threadIdx.x >> 6, f = threadIdx.x & 63;
  float s = 0.f;
  for (int c = g; c < a.nchunk; c += 4) s += a.part[j][(int64_t)c * H + f];
  red[g][f] = s;
  __syncthreads();
  if (g == 0) a.out[j][f] = ((red[0][f] + red[1][f]) + red[2][f]) + red[3][f];
}

// G1 = (T2 W2a) * dropout-mask * [H1 > 0]; partial column sums for db1.  The forward kept
// A1 = dropout(relu(H1)): A1 > 0 exactly where the mask kept a positive H1, so no Philox here.
// CTA = BM_ROWS rows: 8 warps x 8 row pairs, half-warp per row.
__global__ void __launch_bounds__(256) k_bwd_mix(BwdMixArgs a) {
  __shared__ __align__(16) float sW[H * H];   // [o][k] = W2[o][k], k < 64
  __shared__ __align__(16) float sT[16][2 * H];   // two T2 rows per half-warp (matvec2_smem)
  __shared__ float red[16][H];
  const BwdMixDir& p = a.d[blockIdx.y];
  for (int i = threadIdx.x; i < H * H; i += blockDim.x) sW[i] = p.w2[(int64_t)(i >> 6) * a.ldw2 + (i & 63)];
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, sub = lane & 15, half = lane >> 4;
  const unsigned hm = half_mask(half);
  float* scratch = sT[threadIdx.x >> 4];
  const int64_t base = (int64_t)blockIdx.x * BM_ROWS + w * 16;
  float4 cs = make_float4(0.f, 0.f, 0.f, 0.f);
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int r = 0; r < 8; r += 2) {   // rows in ascending order per half-warp, two per pass over W2a
    const int64_t i0 = base + 2 * r + half, i1 = i0 + 2;
    const bool ok0 = i0 < a.N, ok1 = i1 < a.N;
    const float4 t0 = ok0 ? ld4(p.t2 + i0 * H + 4 * sub) : zero;
    const float4 t1 = ok1 ? ld4(p.t2 + i1 * H + 4 * sub) : zero;
    const float4 h0 = ok0 ? ld4(p.h1 + i0 * H + 4 * sub) : zero;
    const float4 h1 = ok1 ? ld4(p.h1 + i1 * H + 4 * sub) : zero;
    float4 g0, g1;
    matvec2_smem(t0, t1, sW, scratch, sub, hm, g0, g1);
    const float sc = p.drop.on ? p.drop.scale : 1.f;   // x 1.0f is exact
    g0.x = h0.x > 0.f ? __fmul_rn(g0.x, sc) : 0.f;
    g0.y = h0.y > 0.f ? __fmul_rn(g0.y, sc) : 0.f;
    g0.z = h0.z > 0.f ? __fmul_rn(g0.z, sc) : 0.f;
    g0.w = h0.w > 0.f ? __fmul_rn(g0.w, sc) : 0.f;
    g1.x = h1.x > 0.f ? __fmul_rn(g1.x, sc) : 0.f;
    g1.y = h1.y > 0.f ? __fmul_rn(g1.y, sc) : 0.f;
    g1.z = h1.z > 0.f ? __fmul_rn(g1.z, sc) : 0.f;
    g1.w = h1.w > 0.f ? __fmul_rn(g1.w, sc) : 0.f;
    if (ok0) st4(p.g1 + i0 * H + 4 * sub, g0);
    if (ok1) st4(p.g1 + i1 * H + 4 * sub, g1);
    cs.x += g0.x; cs.y += g0.y; cs.z += g0.z; cs.w += g0.w;
    cs.x += g1.x; cs.y += g1.y; cs.z += g1.z; cs.w += g1.w;
  }
  st4(&red[w * 2 + half][4 * sub], cs);
  __syncthreads();
  if (threadIdx.x < H) {
    float s = 0.f;
#pragma unroll
    for (int q = 0; q < 16; ++q) s += red[q][threadIdx.x];
    p.part[(int64_t)blockIdx.x * H + threadIdx.x] = s;
  }
}


// C[o][k] = sum_i U[i][o] * V[i][k]  (64 x 64), rows chunked; partial[chunk][64*64]
__global__ void __launch_bounds__(256) k_outer64(OuterArgs a) {
  __shared__ __align__(16) float sU[64][H];
  __shared__ __align__(16) float sV[64][H];
  const int d = blockIdx.y;
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
  const int64_t base = (int64_t)blockIdx.x * OP_ROWS;
  const int64_t end = min(a.N, base + OP_ROWS);
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int64_t r0 = base; r0 < end; r0 += 64) {
    const int nr = (int)min((int64_t)64, end - r0);
    for (int i = threadIdx.x; i < 64 * H / 4; i += 256) {
      const int r = i >> 4, c4 = i & 15;
      float4 uv = make_float4(0.f, 0.f, 0.f, 0.f), vv = uv;
      if (r < nr) {
        uv = *reinterpret_cast<const float4*>(a.u[d] + (r0 + r) * H + c4 * 4);
        vv = *reinterpret_cast<const float4*>(a.v[d] + (r0 + r) * H + c4 * 4);
      }
      *reinterpret_cast<float4*>(&sU[r][c4 * 4]) = uv;
      *reinterpret_cast<float4*>(&sV[r][c4 * 4]) = vv;
    }
    __syncthreads();
#pragma unroll 8
    for (int r = 0; r < 64; ++r) {
      const float4 u4 = *reinterpret_cast<const float4*>(&sU[r][ty * 4]);
      const float4 v4 = *reinterpret_cast<const float4*>(&sV[r][tx * 4]);
      const float uu[4] = {u4.x, u4.y, u4.z, u4.w};
      const float vv[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        fma2(acc[i][0], acc[i][1], uu[i], vv[0], vv[1]);
        fma2(acc[i][2], acc[i][3], uu[i], vv[2], vv[3]);
      }
    }
    __syncthreads();
  }
  float* out = a.part[d] + (int64_t)blockIdx.x * H * H;
#pragma unroll
  for (int i = 0; i < 4; ++i)
    *reinterpret_cast<float4*>(out + (ty * 4 + i) * H + tx * 4) =
        make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
}
// dst[o*ld + k] = sum_chunk part[chunk][o*64 + k]: CTA = 64 outputs x 4 chains (chain g takes
// the chunks c = g mod 4 in order, 8 loads in flight), combined as (s0 + s1) + (s2 + s3)
__global__ void __launch_bounds__(256) k_outer_reduce(OuterReduceArgs a) {
  __shared__ float red[4][64];
  const int d = blockIdx.y;
  const int g = threadIdx.x >> 6, l = threadIdx.x & 63;
  const int idx = blockIdx.x * 64 + l;  // 0..4095
  const float* __restrict__ p = a.part[d] + idx;
  float s = 0.f;
  int c = g;
  for (; c + 28 < a.nchunk; c += 32) {
    float v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = p[(int64_t)(c + 4 * u) * H * H];
#pragma unroll
    for (int u = 0; u < 8; ++u) s += v[u];
  }
  for (; c < a.nchunk; c += 4) s += p[(int64_t)c * H * H];
  red[g][l] = s;
  __syncthreads();
  if (g == 0) a.dst[d][(int64_t)(idx >> 6) * a.ld + (idx & 63)] = (red[0][l] + red[1][l]) + (red[2][l] + red[3][l]);
}

// per-tree segment sum: dP[d][b][f] = sum_{i in b} T2_d[i][f]   (eval-mode dW2b)
__global__ void __launch_bounds__(256) k_segsum(SegSumArgs a) {
  __shared__ float part[4][H];
  const int d = blockIdx.y;
  const int64_t b = blockIdx.x;
  const int g = threadIdx.x >> 6, f = threadIdx.x & 63;
  const int s = a.node_ptr[b], e = a.node_ptr[b + 1];
  float acc = 0.f;
  for (int i = s + g; i < e; i += 4) acc += a.t[d][(int64_t)i * H + f];
  part[g][f] = acc;
  __syncthreads();
  if (g == 0) a.out[d][b * H + f] = ((part[0][f] + part[1][f]) + part[2][f]) + part[3][f];
}

// dW2[o][64 + k] for one column k per CTA (4 warps):
//   train: scale * sum_b relu(x_root_b[k]) * sum_{i in b} keep(i, 64+k) * T2[i][o]
//   eval : sum_b relu(x_root_b[k]) * dP[b][o]
// Trees ascending, rows ascending inside a warp's strip, warps combined in order.
__global__ void __launch_bounds__(128) k_dw2b(Dw2bArgs a) {
  if (*a.overflow == 0) return;   // sparse roots: the (part, reduce) pair below did the work
  __shared__ float red[4][H];
  __shared__ int s_hit_b[128];
  __shared__ float s_hit_v[128];
  __shared__ int s_nhit;
  const Dw2bDir& p = a.d[blockIdx.y];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int64_t k = blockIdx.x; k < a.K; k += gridDim.x) {   // columns round-robin over a capped grid
  float2 acc = make_float2(0.f, 0.f);
  const uint32_t c = (uint32_t)(H + k);
  for (int64_t b0 = 0; b0 < a.B; b0 += 128) {
    // ordered hit list of this group of 128 trees (warp 0 compacts in tree order)
    __syncthreads();
    if (w == 0) {
      int n = 0;
      for (int q = 0; q < 4; ++q) {
        const int64_t b = b0 + q * 32 + lane;
        float v = 0.f;
        if (b < a.B) {   // relu(x_root[b][k]) through the slot map (no dense x needed)
          const int t = a.slot[k * a.B + b];
          if (t >= 0) v = a.rnz_val[b * a.K + t];
        }
        const unsigned m = __ballot_sync(FULL_MASK, v > 0.f);
        if (v > 0.f) {
          const int pos = n + __popc(m & ((1u << lane) - 1u));
          s_hit_b[pos] = (int)b;
          s_hit_v[pos] = v;
        }
        n += __popc(m);
      }
      if (lane == 0) s_nhit = n;
    }
    __syncthreads();
    const int nhit = s_nhit;
    for (int hI = 0; hI < nhit; ++hI) {
      const int b = s_hit_b[hI];
      const float v = s_hit_v[hI];
      if (p.drop.on) {
        const int s = a.node_ptr[b], e = a.node_ptr[b + 1];
        float2 sub = make_float2(0.f, 0.f);
        for (int i0 = s + w * 32; i0 < e; i0 += 128) {
          const int i = i0 + lane;
          bool keep = false;
          if (i < e) {
            const Philox4 r = drop_block(p.drop, a.node_id_base + i, c >> 2);
            keep = philox_elem(r, c & 3) >= p.drop.thresh;
          }
          unsigned m = __ballot_sync(FULL_MASK, keep);
          while (m) {
            const int sl = __ffs(m) - 1;
            m &= m - 1;
            const float2 t = *reinterpret_cast<const float2*>(p.t2 + (int64_t)(i0 + sl) * H + 2 * lane);
            sub.x += t.x;
            sub.y += t.y;
          }
        }
        acc.x = fmaf(v, sub.x, acc.x);
        acc.y = fmaf(v, sub.y, acc.y);
      } else if (w == 0) {
        const float2 t = *reinterpret_cast<const float2*>(p.dP + (int64_t)b * H + 2 * lane);
        acc.x = fmaf(v, t.x, acc.x);
        acc.y = fmaf(v, t.y, acc.y);
      }
    }
  }
  red[w][2 * lane] = acc.x;
  red[w][2 * lane + 1] = acc.y;
  __syncthreads();
  if (threadIdx.x < H) {
    const float s = ((red[0][threadIdx.x] + red[1][threadIdx.x]) + red[2][threadIdx.x]) + red[3][threadIdx.x];
    p.dw2[(int64_t)threadIdx.x * a.ld + H + k] = p.drop.on ? s * p.drop.scale : s;
  }
  __syncthreads();   // red[] is reused by the next column
  }
}

// ---- dW2b, sparse-root fast path (every root row has <= DW2B_CAP positive columns) -----
// part: CTA = DW2B_ROWS consecutive rows of the batch, T2 rows staged in shared memory.
//   For every tree segment in the block and every root slot t of that tree (warps take
//   slots round-robin): S[(blk + b)][t][:] = sum_{i in segment, keep(i, 64 + col_t)} T2[i][:]
//   (lanes decide keep for 32 rows with one Philox block each, then add the kept rows).
//   (blk + b) is unique per (block, tree) pair because trees are contiguous and sorted.
// reduce: warp per column k: trees ascending (slot map), blocks ascending:
//   dW2[o][64 + k] = scale * sum_b relu(x_root_b[k]) * sum_blk S[(blk + b)][slot][o]
//   eval / p = 0:   dW2[o][64 + k] = sum_b relu(x_root_b[k]) * dP[b][o]
static_assert(DW2B_CAP <= 64, "the forward hands the keep decisions over as one 64-bit word per node");
__global__ void __launch_bounds__(256) k_dw2b_part(Dw2bArgs a) {
  if (*a.overflow != 0) return;
  __shared__ __align__(16) float sT[DW2B_ROWS * H];
  __shared__ unsigned long long sK[DW2B_ROWS];   // the forward's keep decisions per (row, root slot)
  const Dw2bDir& p = a.d[blockIdx.y];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t r0 = (int64_t)blockIdx.x * DW2B_ROWS;
  const int64_t r1 = min(a.N, r0 + DW2B_ROWS);
  if (threadIdx.x < DW2B_ROWS) sK[threadIdx.x] = r0 + threadIdx.x < r1 ? p.keep[r0 + threadIdx.x] : 0ull;
  for (int i = threadIdx.x; i < DW2B_ROWS * H / 4; i += 256) {
    const int64_t r = r0 + (i >> 4);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < r1) v = *reinterpret_cast<const float4*>(p.t2 + r * H + (i & 15) * 4);
    *reinterpret_cast<float4*>(sT + (size_t)i * 4) = v;
  }
  __syncthreads();
  const int64_t b_first = a.batch[r0], b_last = a.batch[r1 - 1];
  for (int64_t b = b_first; b <= b_last; ++b) {
    const int s = max((int)r0, a.node_ptr[b]), e = min((int)r1, a.node_ptr[b + 1]);
    if (s >= e) continue;
    const int cnt = a.rnz_cnt[b];
    float* Sb = p.S + ((size_t)(blockIdx.x + b) * DW2B_CAP) * H;
    for (int t = w; t < cnt; t += 8) {
      float2 acc = make_float2(0.f, 0.f);
      for (int i0 = s; i0 < e; i0 += 32) {
        const int i = i0 + lane;
        const bool keep = i < e && ((sK[i - r0] >> t) & 1ull);   // t < DW2B_CAP = 64 on this path
        unsigned m = __ballot_sync(FULL_MASK, keep);
        while (m) {
          const int sl = __ffs(m) - 1;
          m &= m - 1;
          const float2 tv = *reinterpret_cast<const float2*>(sT + (size_t)(i0 + sl - r0) * H + 2 * lane);
          acc.x += tv.x;
          acc.y += tv.y;
        }
      }
      *reinterpret_cast<float2*>(Sb + (size_t)t * H + 2 * lane) = acc;
    }
  }
}

__global__ void __launch_bounds__(256) k_dw2b_reduce(Dw2bArgs a) {
  if (*a.overflow != 0) return;
  // CTA = 2 columns x 4 warps; warp g of a column takes the 32-tree rounds r = g, g+4, ...;
  // the four partial sums are combined in warp order.
  __shared__ float red[2][4][H];
  const Dw2bDir& p = a.d[blockIdx.y];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int cg = w >> 2, g = w & 3;
  for (int64_t kp = blockIdx.x; kp * 2 < a.K; kp += gridDim.x) {   // column pairs (CTA launch rate, not work, bound this)
  const int64_t k = kp * 2 + cg;
  float2 acc = make_float2(0.f, 0.f);
  // most columns are positive in no root row of the batch: nothing to look up for them
  if (k < a.K && a.overflow[1 + k] != 0) {
    for (int64_t b0 = (int64_t)g * 32; b0 < a.B; b0 += 128) {
      const int64_t b = b0 + lane;
      const int t = b < a.B ? a.slot[k * a.B + b] : -1;   // column-major: one coalesced load per 32 trees
      float v = 0.f;
      int s = 0, e = 0;
      if (t >= 0) {                       // lanes fetch their tree's operands in parallel
        v = a.rnz_val[b * a.K + t];
        s = a.node_ptr[b];
        e = a.node_ptr[b + 1];
      }
      unsigned m = __ballot_sync(FULL_MASK, t >= 0);
      while (m) {
        const int sl = __ffs(m) - 1;
        m &= m - 1;
        const int64_t bb = b0 + sl;
        const int tt = __shfl_sync(FULL_MASK, t, sl);
        const float vv = __shfl_sync(FULL_MASK, v, sl);
        float2 sub = make_float2(0.f, 0.f);
        if (p.drop.on) {
          const int ss = __shfl_sync(FULL_MASK, s, sl), ee = __shfl_sync(FULL_MASK, e, sl);
          if (ee > ss) {
            const int j0 = ss / DW2B_ROWS, j1 = (ee - 1) / DW2B_ROWS;
            for (int j = j0; j <= j1; ++j) {
              const float2 q = *reinterpret_cast<const float2*>(
                  p.S + ((size_t)(j + bb) * DW2B_CAP + tt) * H + 2 * lane);
              sub.x += q.x;
              sub.y += q.y;
            }
          }
        } else {
          sub = *reinterpret_cast<const float2*>(p.dP + bb * H + 2 * lane);
        }
        acc.x = fmaf(vv, sub.x, acc.x);
        acc.y = fmaf(vv, sub.y, acc.y);
      }
    }
  }
  red[cg][g][2 * lane] = acc.x;
  red[cg][g][2 * lane + 1] = acc.y;
  __syncthreads();
  if (g == 0 && k < a.K) {
    const float sc = p.drop.on ? p.drop.scale : 1.f;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int o = 2 * lane + h;
      const float tot = ((red[cg][0][o] + red[cg][1][o]) + red[cg][2][o]) + red[cg][3][o];
      p.dw2[(int64_t)o * a.ld + H + k] = tot * sc;
    }
  }
  __syncthreads();
  }
}

// ---------------------------------------------------------------- dropout mask materialisation (tests)
__global__ void k_dropout_mask(DropSpec ds, int64_t node_id_base, int64_t N, int64_t n_cols,
                               uint8_t* keep) {
  const int64_t nblk = (n_cols + 3) / 4;
  const int64_t tot = N * nblk;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < tot;
       t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = t / nblk, blk = t % nblk;
    const Philox4 r = drop_block(ds, node_id_base + i, (uint32_t)blk);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int64_t c = blk * 4 + e;
      if (c < n_cols) keep[i * n_cols + c] = philox_elem(r, e) >= ds.thresh ? 1 : 0;
    }
  }
}

// ---------------------------------------------------------------- host-side launchers
int root_nz_csr_launch(const RootNzArgs& a, const int32_t* xptr, const int32_t* xcol, const float* xval,
                       cudaStream_t st) {
  cudaMemsetAsync(a.overflow, 0, (size_t)(1 + a.K) * sizeof(int32_t), st);
  if (a.B == 0) return 0;
  cudaMemsetAsync(a.slot, 0xFF, (size_t)a.B * a.K * sizeof(int32_t), st);   // -1: column not positive in that root
  k_root_nz_csr<<<(int)a.B, 256, 0, st>>>(a, xptr, xcol, xval);
  BIGCN_CHECK_LAUNCH("k_root_nz_csr");
  return 0;
}
int root_nz_launch(const RootNzArgs& a, cudaStream_t st) {
  cudaMemsetAsync(a.overflow, 0, (size_t)(1 + a.K) * sizeof(int32_t), st);
  if (a.B == 0) return 0;
  cudaMemsetAsync(a.slot, 0xFF, (size_t)a.B * a.K * sizeof(int32_t), st);   // -1: column not positive in that root
  const size_t smem = (size_t)((a.K + 31) / 32) * sizeof(int);
  BIGCN_CHECK_ARG(smem <= 48 * 1024, "root_nz: in_feats too large (%lld)", (long long)a.K);
  if (a.x_bf16) k_root_nz<__nv_bfloat16><<<(int)a.B, 256, smem, st>>>(a);
  else k_root_nz<float><<<(int)a.B, 256, smem, st>>>(a);
  BIGCN_CHECK_LAUNCH("k_root_nz");
  return 0;
}
int root_proj_launch(const RootProjArgs& a, int ndir, cudaStream_t st) {
  if (a.B == 0) return 0;
  k_root_proj<<<dim3((int)ceil_div(a.B, 8), ndir), 256, 0, st>>>(a);
  BIGCN_CHECK_LAUNCH("k_root_proj");
  return 0;
}
template <int R, int Q, int MINB>
static int mix_launch(const MixArgs& a0, int ndir, cudaStream_t st) {
  constexpr int smem = SweepSmem<R, Q>::kBytes;
  static bool attr = false;
  if (!attr) {
    sweep_attr(k_prop1_mix<R, Q, MINB>, smem);
    attr = true;
  }
  MixArgs a = a0;
  const int max_ctas = num_sms() * MINB;
  a.cb = sweep_cb(a.N, R, max_ctas);
  k_prop1_mix<R, Q, MINB><<<dim3(sweep_grid(a.N, R, a.cb, max_ctas), ndir), 256, smem, st>>>(a);
  BIGCN_CHECK_LAUNCH("k_prop1_mix");
  return 0;
}
int prop1_mix_launch(const MixArgs& a, int ndir, cudaStream_t st, const EntryW* ew) {
  if (a.N == 0) return 0;
  if (ew) {   // one configuration, the default one
    constexpr int smem = SweepSmem<MIX_R, MIX_Q>::kBytes;
    static bool attr = false;
    if (!attr) {
      sweep_attr(k_prop1_mix_w, smem);
      attr = true;
    }
    MixArgs m = a;
    const int max_ctas = num_sms() * 4;
    m.cb = sweep_cb(m.N, MIX_R, max_ctas);
    k_prop1_mix_w<<<dim3(sweep_grid(m.N, MIX_R, m.cb, max_ctas), ndir), 256, smem, st>>>(m, *ew);
    BIGCN_CHECK_LAUNCH("k_prop1_mix_w");
    return 0;
  }
  switch (debug_knob(2)) {
    case 1: return mix_launch<4, 4, 4>(a, ndir, st);
    case 2: return mix_launch<2, 8, 4>(a, ndir, st);
    case 3: return mix_launch<2, 4, 5>(a, ndir, st);
    case 4: return mix_launch<8, 8, 2>(a, ndir, st);
    case 5: return mix_launch<4, 8, 3>(a, ndir, st);
    default: return mix_launch<MIX_R, MIX_Q, 4>(a, ndir, st);
  }
}
size_t readout_scratch_floats(int64_t N, int64_t B, int ndir) {
  return (size_t)ndir * (size_t)(ceil_div(N > 0 ? N : 1, RO_SLICE) + B) * 2 * H;
}
int readout_launch(const ReadoutArgs& a0, cudaStream_t st, bool with_final) {
  if (a0.B == 0) return 0;
  ReadoutArgs a = a0;
  a.nitems = ceil_div(a.N > 0 ? a.N : 1, RO_SLICE) + a.B;
  if (a.N > 0) {
    k_readout_part<<<dim3((unsigned)a.nitems, a.ndir), 256, 0, st>>>(a);
    BIGCN_CHECK_LAUNCH("k_readout_part");
  }
  if (!with_final) return 0;       // the fused tail (k_train_tail) finishes the trees
  k_readout_final<<<(int)ceil_div(a.B, 4), 256, 0, st>>>(a);
  BIGCN_CHECK_LAUNCH("k_readout_final");
  return 0;
}
int cs_chunks(int64_t N) { return (int)ceil_div(N > 0 ? N : 1, CS_ROWS); }
int gs_chunks(int64_t B) { return (int)ceil_div(B > 0 ? B : 1, GS_TREES); }
int bm_chunks(int64_t N) { return (int)ceil_div(N > 0 ? N : 1, BM_ROWS); }
int op_chunks(int64_t N) { return (int)ceil_div(N > 0 ? N : 1, OP_ROWS); }

int gscale_launch(const GScaleArgs& a, int ndir, cudaStream_t st) {
  if (a.B == 0) return 0;
  k_gscale<<<dim3(gs_chunks(a.B), ndir), 256, 0, st>>>(a);
  BIGCN_CHECK_LAUNCH("k_gscale");
  return 0;
}
int propagate_g2_launch(const PropG2Args& a0, int ndir, cudaStream_t st, const EntryW* ew) {
  if (a0.N == 0) return 0;
  constexpr int smem = SweepSmem<PROP_R, PROP_Q>::kBytes;
  static bool attr = false;
  if (!attr) {
    sweep_attr(k_propagate_g2, smem);
    sweep_attr(k_propagate_g2_w, smem);
    attr = true;
  }
  PropG2Args a = a0;
  const int max_ctas = num_sms() * 3;
  a.cb = sweep_cb(a.N, PROP_R, max_ctas);
  const dim3 grid(sweep_grid(a.N, PROP_R, a.cb, max_ctas), ndir);
  if (ew) {
    k_propagate_g2_w<<<grid, 256, smem, st>>>(a, *ew);
    BIGCN_CHECK_LAUNCH("k_propagate_g2_w");
    return 0;
  }
  k_propagate_g2<<<grid, 256, smem, st>>>(a);
  BIGCN_CHECK_LAUNCH("k_propagate_g2");
  return 0;
}
int colsum_reduce_launch(const ColsumArgs& a, int njobs, cudaStream_t st) {
  k_colsum_reduce<<<njobs, 256, 0, st>>>(a);
  BIGCN_CHECK_LAUNCH("k_colsum_reduce");
  return 0;
}
int bwd_mix_launch(const BwdMixArgs& a, int ndir, cudaStream_t st) {
  if (a.N == 0) return 0;
  k_bwd_mix<<<dim3(bm_chunks(a.N), ndir), 256, 0, st>>>(a);
  BIGCN_CHECK_LAUNCH("k_bwd_mix");
  return 0;
}
int outer64_launch(const OuterArgs& a, const OuterReduceArgs& r, int ndir, cudaStream_t st) {
  if (a.N > 0) {
    k_outer64<<<dim3(op_chunks(a.N), ndir), 256, 0, st>>>(a);
    BIGCN_CHECK_LAUNCH("k_outer64");
  }
  k_outer_reduce<<<dim3(H * H / 64, ndir), 256, 0, st>>>(r);
  BIGCN_CHECK_LAUNCH("k_outer_reduce");
  return 0;
}
int segsum_launch(const SegSumArgs& a, int64_t B, int ndir, cudaStream_t st) {
  if (B == 0) return 0;
  k_segsum<<<dim3((int)B, ndir), 256, 0, st>>>(a);
  BIGCN_CHECK_LAUNCH("k_segsum");
  return 0;
}
int dw2b_launch(const Dw2bArgs& a, int ndir, bool dropping, cudaStream_t st) {
  if (a.K == 0) return 0;
  if (dropping && a.N > 0) {
    k_dw2b_part<<<dim3(dw2b_blocks(a.N), ndir), 256, 0, st>>>(a);
    BIGCN_CHECK_LAUNCH("k_dw2b_part");
  }
  {
    int64_t g = ceil_div(a.K, 2);
    const int64_t cap = (int64_t)num_sms() * 4;
    if (g > cap) g = cap;
    k_dw2b_reduce<<<dim3((int)g, ndir), 256, 0, st>>>(a);
  }
  BIGCN_CHECK_LAUNCH("k_dw2b_reduce");
  {   // dense-root fallback, returns at once otherwise (a capped grid: the usual case is 1 k CTAs that exit)
    int64_t g = a.K;
    const int64_t cap = (int64_t)num_sms() * 8;
    if (g > cap) g = cap;
    k_dw2b<<<dim3((int)g, ndir), 128, 0, st>>>(a);
  }
  BIGCN_CHECK_LAUNCH("k_dw2b");
  return 0;
}
int dw2b_blocks(int64_t N) { return (int)ceil_div(N > 0 ? N : 1, DW2B_ROWS); }
int dropout_mask_launch(const DropSpec& ds, int64_t base, int64_t N, int64_t n_cols, uint8_t* keep,
                        cudaStream_t st) {
  if (N == 0 || n_cols == 0) return 0;
  k_dropout_mask<<<num_sms() * 4, 256, 0, st>>>(ds, base, N, n_cols, keep);
  BIGCN_CHECK_LAUNCH("k_dropout_mask");
  return 0;
}

}  // namespace bigcn
