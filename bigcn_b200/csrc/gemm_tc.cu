// tcgen05 / TMA / TMEM GEMM for the feature transform  Y[N, n_out] = X[N, K] * W^T.
//
// Replaces GCNConv.lin (cuBLAS SGEMM) at BiGCN_Twitter.py:42,92 in the tensor-core modes:
//   BIGCN_GEMM_TF32   : one kind::tf32 MMA per K step (operands truncated to TF32 by the MMA)
//   BIGCN_GEMM_TF32X2 : W = W_hi + W_lo with W_lo = W - tf32(W) as a second B operand (two
//                       MMAs per K step); exact to ~2^-22 whenever X is representable in TF32
//                       (bag-of-words counts are)
//   BIGCN_GEMM_TF32X3 : X is split as well: four converter warps rewrite every X tile in shared memory
//                       as X_hi (in place) and X_lo (a sibling buffer with the same swizzle) between the TMA
//                       load and the MMA, three MMAs per K step (X_hi W_hi + X_hi W_lo + X_lo W_hi):
//                       fp32-class accuracy on dense signed features, X still read from HBM once
// Both operands are K-major exactly as they sit in HBM: X is [N, K] row-major and the PyG
// weights are [64, K] row-major, so TMA loads them straight into 128B-swizzled shared memory
// (no transposed copy).  The TD and BU weights are two 64-row boxes of one B tile, so X is
// read ONCE for both directions.  One CTA owns 256 rows of X: two M=128 accumulators in TMEM
// share every B tile, halving the L2 traffic for W.  Warp-specialised, mbarrier ring:
//   warp 0 : TMA producer            warp 1 : tcgen05.mma issuer (one elected lane)
//   warp 2 : TMEM allocator          warps 4-7 : epilogue (tcgen05.ld -> registers -> HBM)
// The kernel is HBM-bound on X (64 flop/B at n_out = 128 < the TF32 ridge).
#include "tc.cuh"

namespace bigcn {

constexpr int TC_BLOCK_M = 256;
constexpr int TC_BLOCK_K = 32;                      // 32 fp32 = 128 B = one swizzle atom
constexpr int TC_UMMA_K = 8;                        // kind::tf32
constexpr int TC_A_BYTES = TC_BLOCK_M * 128;        // 32 KB
constexpr int TC_THREADS = 256;
constexpr int TC_THREADS_XS = 384;                  // + warps 8..11: X hi/lo converters (TF32X3)

struct TcParams {
  float* y;
  int64_t ldy;
  int64_t N, K;
  int n_out;       // 64 or 128
  int num_tiles;   // ceil(N / 256)
  int num_kb;      // ceil(K / 32)
  // split-K for small N (a PHEME batch of 24 trees is ONE 256-row tile: one SM would walk all K blocks alone):
  // grid.y CTAs take kb_per K blocks each and write partial[y][row][n_out]; k_xw_splitk_reduce adds them in order
  int kb_per;      // K blocks per CTA (= num_kb when not split)
  float* partial;  // [grid.y][N][n_out] or NULL
};

// Epilogue warps 4..7 of k_xw_tc / k_xw_bf16 (q = TMEM lane quarter this warp may access): per tile, the two M = 128
// accumulators TMEM -> registers -> y (or this split's partial), then hand TMEM back to the MMA issuer
__device__ __forceinline__ void xw_epilogue(const TcParams& p, uint32_t tmem_base, uint32_t bar_tmem_full,
                                            uint32_t bar_tmem_empty, int q, int lane) {
  uint32_t tile_ph = 0;
  for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, tile_ph ^= 1) {
    mbar_wait(bar_tmem_full, tile_ph);
    tc_fence_after();
    const int64_t m0 = (int64_t)tile * TC_BLOCK_M;
#pragma unroll 1
    for (int a = 0; a < 2; ++a) {
      const int64_t row = m0 + a * 128 + q * 32 + lane;
      for (int c0 = 0; c0 < p.n_out; c0 += 32) {
        uint32_t r[32];
        tc_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(a * 128 + c0), r);
        tc_wait_ld();
        if (row < p.N) {
          float4* dst = p.partial ? reinterpret_cast<float4*>(p.partial + ((int64_t)blockIdx.y * p.N + row) * p.n_out + c0)
                                  : reinterpret_cast<float4*>(p.y + row * p.ldy + c0);
#pragma unroll
          for (int j = 0; j < 8; ++j)
            dst[j] = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]),
                                 __uint_as_float(r[4 * j + 2]), __uint_as_float(r[4 * j + 3]));
        }
      }
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(bar_tmem_empty);
  }
}

// NB = number of B operands per stage (1: W, 2: W and W_lo); XS: X split hi / lo in shared memory (TF32X3)
template <int NB, bool XS>
__global__ void __launch_bounds__(XS ? TC_THREADS_XS : TC_THREADS, 1)
k_xw_tc(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w0,
        const __grid_constant__ CUtensorMap map_w1, const __grid_constant__ CUtensorMap map_l0,
        const __grid_constant__ CUtensorMap map_l1, const TcParams p) {
  static_assert(!XS || NB == 2, "the X split goes with the W split");
  constexpr int STAGES = XS ? 2 : (NB == 1 ? 4 : 3);
  constexpr int A_SLOTS = XS ? 2 : 1;                          // [X | X_lo]
  extern __shared__ __align__(1024) uint8_t tc_smem[];
  const int b_bytes = p.n_out * 128;                           // one B operand tile
  constexpr int B_OFF = A_SLOTS * TC_A_BYTES;
  constexpr int stage_bytes = B_OFF + NB * 16384;              // B slots are 16 KB apart (1024 B aligned)
  __shared__ __align__(8) uint64_t bar_full[STAGES];
  __shared__ __align__(8) uint64_t bar_conv[STAGES];           // XS: the stage's X tile is split (4 converter warps)
  __shared__ __align__(8) uint64_t bar_empty[STAGES];
  __shared__ __align__(8) uint64_t bar_tmem_full, bar_tmem_empty;
  __shared__ uint32_t tmem_base_s;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // 1024 B alignment of the dynamic region (SWIZZLE_128B atoms)
  const uint32_t smem0 = (smem_u32(tc_smem) + 1023u) & ~1023u;
  const int kb0 = blockIdx.y * p.kb_per, kb1 = min(p.num_kb, kb0 + p.kb_per);   // this CTA's K blocks (split-K: grid.y > 1)

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_x);
    tma_prefetch_desc(&map_w0);
    if (p.n_out == 128) tma_prefetch_desc(&map_w1);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(smem_u32(&bar_full[s]), 1);
      mbar_init(smem_u32(&bar_empty[s]), 1);
      mbar_init(smem_u32(&bar_conv[s]), 4);
    }
    mbar_init(smem_u32(&bar_tmem_full), 1);
    mbar_init(smem_u32(&bar_tmem_empty), 4);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {   // 256 TMEM columns: two fp32 accumulators of up to 128 columns
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(smem_u32(&tmem_base_s)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp == 0) {
    if (lane == 0) {   // ===== TMA producer =====
      int s = 0;
      uint32_t ph = 0;
      const uint32_t tx = (uint32_t)(TC_A_BYTES + NB * b_bytes);
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        const int m0 = tile * TC_BLOCK_M;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(smem_u32(&bar_empty[s]), ph ^ 1);
          const uint32_t full = smem_u32(&bar_full[s]);
          const uint32_t sa = smem0 + s * stage_bytes;
          mbar_expect_tx(full, tx);
          tma_load_2d(sa, &map_x, full, kb * TC_BLOCK_K, m0);
          tma_load_2d(sa + B_OFF, &map_w0, full, kb * TC_BLOCK_K, 0);
          if (p.n_out == 128) tma_load_2d(sa + B_OFF + 64 * 128, &map_w1, full, kb * TC_BLOCK_K, 0);
          if (NB == 2) {
            tma_load_2d(sa + B_OFF + 16384, &map_l0, full, kb * TC_BLOCK_K, 0);
            if (p.n_out == 128) tma_load_2d(sa + B_OFF + 16384 + 64 * 128, &map_l1, full, kb * TC_BLOCK_K, 0);
          }
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {   // ===== MMA issuer =====
      const uint32_t idesc = make_idesc_tf32(128, p.n_out);
      int s = 0;
      uint32_t ph = 0, tile_ph = 0;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, tile_ph ^= 1) {
        mbar_wait(smem_u32(&bar_tmem_empty), tile_ph ^ 1);   // epilogue has drained the accumulators
        tc_fence_after();
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(smem_u32(XS ? &bar_conv[s] : &bar_full[s]), ph);
          tc_fence_after();
          const uint32_t sa = smem0 + s * stage_bytes;
#pragma unroll
          for (int k = 0; k < TC_BLOCK_K / TC_UMMA_K; ++k) {
            const uint32_t koff = k * TC_UMMA_K * 4;           // 32 B per K step inside the 128 B atom
            const uint64_t da0 = make_desc_k_sw128(sa + koff);
            const uint64_t da1 = make_desc_k_sw128(sa + 128 * 128 + koff);
            const uint64_t db = make_desc_k_sw128(sa + B_OFF + koff);
            const uint32_t acc = ((kb - kb0) | k) ? 1u : 0u;
            tc_mma_tf32(tmem_base, da0, db, idesc, acc);
            tc_mma_tf32(tmem_base + 128, da1, db, idesc, acc);
            if (NB == 2) {
              const uint64_t dl = make_desc_k_sw128(sa + B_OFF + 16384 + koff);
              tc_mma_tf32(tmem_base, da0, dl, idesc, 1u);
              tc_mma_tf32(tmem_base + 128, da1, dl, idesc, 1u);
            }
            if (XS) {                                          // X_lo * W_hi
              const uint64_t dx0 = make_desc_k_sw128(sa + TC_A_BYTES + koff);
              const uint64_t dx1 = make_desc_k_sw128(sa + TC_A_BYTES + 128 * 128 + koff);
              tc_mma_tf32(tmem_base, dx0, db, idesc, 1u);
              tc_mma_tf32(tmem_base + 128, dx1, db, idesc, 1u);
            }
          }
          tc_commit(smem_u32(&bar_empty[s]));                 // frees the stage when the MMAs retire
          if (kb == kb1 - 1) tc_commit(smem_u32(&bar_tmem_full));
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (XS && warp >= 8) {   // ===== converters: X tile -> X_hi (in place) | X_lo =====
    const int cw = warp - 8;
    int s = 0;
    uint32_t ph = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(smem_u32(&bar_full[s]), ph);
        const uint32_t sa = smem0 + s * stage_bytes;
        split_tile_hi_lo(sa, sa + TC_A_BYTES, TC_A_BYTES, cw, lane);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&bar_conv[s]));
        if (++s == STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp >= 4 && warp < 8) {
    xw_epilogue(p, tmem_base, smem_u32(&bar_tmem_full), smem_u32(&bar_tmem_empty), warp & 3, lane);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem_base));
  }
}

// y[row][c] = sum over the K splits, in split order (deterministic)
__global__ void __launch_bounds__(256) k_xw_splitk_reduce(const float* __restrict__ partial, int nsplit, int64_t N, int n_out,
                                                          float* __restrict__ y, int64_t ldy) {
  const int64_t n4 = N * (n_out / 4);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / (n_out / 4), c4 = i % (n_out / 4);
    float4 acc = reinterpret_cast<const float4*>(partial)[i];
    for (int s = 1; s < nsplit; ++s) {
      const float4 v = reinterpret_cast<const float4*>(partial)[(int64_t)s * n4 + i];
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    *reinterpret_cast<float4*>(y + row * ldy + 4 * c4) = acc;
  }
}

// hi = w with the 13 low mantissa bits cleared (exactly a TF32 value, whatever rounding the MMA
// applies to fp32 operands); lo = tf32(w - hi).  hi + lo == w to ~2^-22 relative.
__global__ void k_split_hi_lo(const float* __restrict__ w, int64_t ldw, int64_t K, float* __restrict__ hi,
                              float* __restrict__ lo) {
  const int64_t n = 64 * K;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float v = w[(i / K) * ldw + (i % K)];
    const float h = __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
    hi[i] = h;
    lo[i] = __uint_as_float((__float_as_uint(v - h) + 0x1000u) & 0xFFFFE000u);   // round to nearest: no sign bias
  }
}

// ---------------------------------------------------------------- host side
bool xw_tc_available() { return encode_fn() != nullptr; }
// BIGCN_GEMM_BF16 (bf16 x; below)
static int xw_bf16(const void* x, int64_t N, int64_t K, const float* const* w, int64_t ldw, int n_out, float* scratch,
                   float* y, int64_t ldy, cudaStream_t st, float* partial);
static int dw_bf16(const void* x, int64_t N, int64_t K, const float* t, int n_out, float* scratch01, float* scratch2,
                   float* partial, float* dw_a, int64_t ldw_a, int64_t k0_a, float* dw_b, int64_t ldw_b, int64_t k0_b,
                   cudaStream_t st);

// w[0], w[1]: the [64, K] PyG weights of the active directions (row pitch ldw); scratch:
// 2 * n_out * K floats for the TF32X3 split (may be NULL in TF32 mode)
size_t xw_tc_partial_floats() { return (size_t)num_sms() * TC_BLOCK_M * 128; }

// few tiles (small batch): split K so that the SMs share the K blocks, at least three per CTA.  Sets p.kb_per and
// p.partial (NULL: not split); returns the number of splits (grid.y)
static int xw_split_k(TcParams& p, float* partial) {
  int nsplit = 1;
  p.kb_per = p.num_kb;
  p.partial = nullptr;
  if (partial != nullptr && p.num_tiles * 4 <= num_sms() && p.num_kb >= 6) {
    int want = num_sms() / p.num_tiles;
    const int max_by_kb = p.num_kb / 3;
    if (want > max_by_kb) want = max_by_kb;
    if (want > 1) {
      p.kb_per = (int)ceil_div(p.num_kb, want);
      nsplit = (int)ceil_div(p.num_kb, p.kb_per);
      if (nsplit > 1) p.partial = partial;
      else p.kb_per = p.num_kb;
    }
  }
  return nsplit;
}

// partial: xw_tc_partial_floats() floats or NULL (no split-K)
int xw_tc_weights(const float* x, int64_t N, int64_t K, const float* const* w, int64_t ldw, int n_out,
                  float* scratch, float* y, int64_t ldy, int mode, cudaStream_t st, float* partial) {
  BIGCN_CHECK_ARG(encode_fn() != nullptr, "xw_tc: cuTensorMapEncodeTiled is unavailable in this driver");
  BIGCN_CHECK_ARG(n_out == 64 || n_out == 128, "xw_tc: n_out must be 64 or 128");
  if (mode == BIGCN_GEMM_BF16) return xw_bf16(x, N, K, w, ldw, n_out, scratch, y, ldy, st, partial);
  BIGCN_CHECK_ARG(K % 4 == 0 && ldw % 4 == 0, "xw_tc: in_feats must be a multiple of 4 for TMA (got %lld)", (long long)K);
  BIGCN_CHECK_ARG((reinterpret_cast<uintptr_t>(x) & 15) == 0, "xw_tc: x must be 16-byte aligned");
  if (N == 0) return 0;
  const int nb = mode == BIGCN_GEMM_TF32 ? 1 : 2;
  const bool xsplit = mode == BIGCN_GEMM_TF32X3;
  BIGCN_CHECK_ARG(nb == 1 || scratch != nullptr, "xw_tc: TF32X2 / TF32X3 need the split scratch");
  CUtensorMap mx, mw0, mw1, ml0, ml1;
  if (int rc = make_map(&mx, x, N, K, K, 256)) return rc;
  if (nb == 1) {
    if (int rc = make_map(&mw0, w[0], 64, K, ldw, 64)) return rc;
    mw1 = mw0;
    if (n_out == 128)
      if (int rc = make_map(&mw1, w[1], 64, K, ldw, 64)) return rc;
    ml0 = mw0;
    ml1 = mw1;
  } else {
    for (int d = 0; d < n_out / 64; ++d) {
      float* hi = scratch + (size_t)(2 * d) * 64 * K;
      float* lo = scratch + (size_t)(2 * d + 1) * 64 * K;
      k_split_hi_lo<<<num_sms() * 2, 256, 0, st>>>(w[d], ldw, K, hi, lo);
      BIGCN_CHECK_LAUNCH("k_split_hi_lo");
      if (int rc = make_map(d == 0 ? &mw0 : &mw1, hi, 64, K, K, 64)) return rc;
      if (int rc = make_map(d == 0 ? &ml0 : &ml1, lo, 64, K, K, 64)) return rc;
    }
    if (n_out == 64) { mw1 = mw0; ml1 = ml0; }
  }
  TcParams p;
  p.y = y; p.ldy = ldy; p.N = N; p.K = K; p.n_out = n_out;
  p.num_tiles = (int)ceil_div(N, TC_BLOCK_M);
  p.num_kb = (int)ceil_div(K, TC_BLOCK_K);
  const int stage_bytes = (xsplit ? 2 : 1) * TC_A_BYTES + nb * 16384;
  const int stages = xsplit ? 2 : (nb == 1 ? 4 : 3);
  const size_t smem = (size_t)stages * stage_bytes + 1024;
  int grid_x = p.num_tiles < num_sms() ? p.num_tiles : num_sms();
  const int nsplit = xw_split_k(p, partial);
  const dim3 grid(grid_x, nsplit);
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(k_xw_tc<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * (TC_A_BYTES + 16384) + 1024);
    cudaFuncSetAttribute(k_xw_tc<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 3 * (TC_A_BYTES + 32768) + 1024);
    cudaFuncSetAttribute(k_xw_tc<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * (2 * TC_A_BYTES + 32768) + 1024);
    attr = true;
  }
  if (nb == 1) k_xw_tc<1, false><<<grid, TC_THREADS, smem, st>>>(mx, mw0, mw1, ml0, ml1, p);
  else if (!xsplit) k_xw_tc<2, false><<<grid, TC_THREADS, smem, st>>>(mx, mw0, mw1, ml0, ml1, p);
  else k_xw_tc<2, true><<<grid, TC_THREADS_XS, smem, st>>>(mx, mw0, mw1, ml0, ml1, p);
  BIGCN_CHECK_LAUNCH("k_xw_tc");
  if (nsplit > 1) {
    int rb = (int)ceil_div(N * (n_out / 4), 256);
    if (rb > num_sms() * 4) rb = num_sms() * 4;
    k_xw_splitk_reduce<<<rb, 256, 0, st>>>(partial, nsplit, N, n_out, y, ldy);
    BIGCN_CHECK_LAUNCH("k_xw_splitk_reduce");
  }
  return 0;
}


// =====================================================================================
// Weight gradient  dW^T[k, o] = sum_i X[i, k] * T[i, o]   (dW1 = T1^T X, SURVEY appendix B)
// as D[M = 128 outputs, N = 256 columns of X] += A^T B over the node axis, kind::tf32.
// Both operands are "MN-major" as they sit in HBM (X[i, :] and T[i, :] are contiguous along
// the M / N axis), which for 32-bit operands is the SWIZZLE_128B_BASE32B shared-memory layout:
// TMA boxes of 32 columns x 32 node rows with CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B.
// Grid = (256-column tiles of X) x (node-range splits), one wave: every CTA streams its slice
// of X exactly once; T (16 MB, L2 resident) is re-read once per column tile.  The accumulator
// (128 x 256 fp32) lives in TMEM; split partials go to partial[split][k][o] and are summed in
// order by k_dw_reduce.  Cost is independent of the sparsity pattern of X.
// NA = 1: T as is (TF32);  NA = 2: T = T_hi + T_lo (fp32-class when X is TF32-exact).
constexpr int DWT_BK = 32;            // node rows per stage
constexpr int DWT_N = 256;            // columns of X per CTA
constexpr int DWT_A_BYTES = 4 * DWT_BK * 128;   // 128 outputs = 4 blocks of 32
constexpr int DWT_B_BYTES = 8 * DWT_BK * 128;   // 256 columns = 8 blocks of 32

// MN-major SWIZZLE_128B_BASE32B descriptor: 128 B (32 fp32) contiguous along MN, rows of the
// K axis 128 B apart, 4-row swizzle atoms (SBO = 512 B), LBO = bytes between 32-element MN blocks
__device__ __forceinline__ uint64_t make_desc_mn_sw128_32b(uint32_t saddr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)(512 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)1 << 61;   // LayoutType::SWIZZLE_128B_BASE32B
  return d;
}
__host__ __device__ constexpr uint32_t make_idesc_tf32_mn(int m, int n) {
  return make_idesc_tf32(m, n) | (1u << 15) | (1u << 16);   // a_major = b_major = MN
}

struct DwtParams {
  float* partial;     // [nsplit][K][n_out]
  int64_t N, K;
  int n_out;
  int rows_per_split; // multiple of DWT_BK
};

// Epilogue warps 4..7 of k_dw_tc / k_dw_bf16: the 128 x 256 accumulator (q < n_out / 32: rows of this direction set)
// TMEM -> registers -> partial[split][col][o]; a CTA without node rows writes zeros
__device__ __forceinline__ void dw_epilogue(const DwtParams& p, uint32_t tmem_base, uint32_t bar_tmem_full, int num_kb,
                                            int col0, int q, int lane) {
  float* out = p.partial + (size_t)blockIdx.y * p.K * p.n_out;
  const int m = q * 32 + lane;
  if (num_kb > 0) {
    mbar_wait(bar_tmem_full, 0);
    tc_fence_after();
  }
  if (q < p.n_out / 32) {
    for (int c0 = 0; c0 < DWT_N; c0 += 32) {
      uint32_t r[32];
      if (num_kb > 0) {
        tc_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, r);
        tc_wait_ld();
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) r[j] = 0u;
      }
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const int64_t col = (int64_t)col0 + c0 + j;
        if (col < p.K) out[col * p.n_out + m] = __uint_as_float(r[j]);   // 32 lanes -> 128 B
      }
    }
  }
}

template <int NA, bool XS>
__global__ void __launch_bounds__(XS ? TC_THREADS_XS : TC_THREADS, 1)
k_dw_tc(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_t,
        const __grid_constant__ CUtensorMap map_tlo, const DwtParams p) {
  static_assert(!XS || NA == 2, "the X split goes with the T split");
  constexpr int STAGES = XS ? 2 : (NA == 1 ? 4 : 3);
  constexpr int STAGE_BYTES = NA * DWT_A_BYTES + (XS ? 2 : 1) * DWT_B_BYTES;   // [T | T_lo | X | X_lo]
  extern __shared__ __align__(1024) uint8_t tc_smem[];
  __shared__ __align__(8) uint64_t bar_full[STAGES];
  __shared__ __align__(8) uint64_t bar_empty[STAGES];
  __shared__ __align__(8) uint64_t bar_conv[STAGES];
  __shared__ __align__(8) uint64_t bar_tmem_full;
  __shared__ uint32_t tmem_base_s;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t smem0 = (smem_u32(tc_smem) + 1023u) & ~1023u;
  const int col0 = blockIdx.x * DWT_N;
  const int64_t r_begin = (int64_t)blockIdx.y * p.rows_per_split;
  const int64_t r_end = min(p.N, r_begin + p.rows_per_split);
  const int num_kb = r_end > r_begin ? (int)((r_end - r_begin + DWT_BK - 1) / DWT_BK) : 0;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_x);
    tma_prefetch_desc(&map_t);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(smem_u32(&bar_full[s]), 1);
      mbar_init(smem_u32(&bar_empty[s]), 1);
      mbar_init(smem_u32(&bar_conv[s]), 4);
    }
    mbar_init(smem_u32(&bar_tmem_full), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(smem_u32(&tmem_base_s)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp == 0) {
    if (lane == 0) {   // ===== TMA producer =====
      int s = 0;
      uint32_t ph = 0;
      // all 4 output blocks are always loaded: blocks beyond n_out are out of bounds -> zero filled
      const uint32_t tx = (uint32_t)(NA * DWT_A_BYTES + DWT_B_BYTES);
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(smem_u32(&bar_empty[s]), ph ^ 1);
        const uint32_t full = smem_u32(&bar_full[s]);
        const uint32_t sa = smem0 + s * STAGE_BYTES;
        const int row = (int)(r_begin + (int64_t)kb * DWT_BK);
        mbar_expect_tx(full, tx);
#pragma unroll
        for (int mb = 0; mb < 4; ++mb) {
          tma_load_2d(sa + mb * (DWT_BK * 128), &map_t, full, mb * 32, row);
          if (NA == 2) tma_load_2d(sa + DWT_A_BYTES + mb * (DWT_BK * 128), &map_tlo, full, mb * 32, row);
        }
#pragma unroll
        for (int nb = 0; nb < 8; ++nb)
          tma_load_2d(sa + NA * DWT_A_BYTES + nb * (DWT_BK * 128), &map_x, full, col0 + nb * 32, row);
        if (++s == STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {   // ===== MMA issuer =====
      const uint32_t idesc = make_idesc_tf32_mn(128, DWT_N);
      int s = 0;
      uint32_t ph = 0;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(smem_u32(XS ? &bar_conv[s] : &bar_full[s]), ph);
        tc_fence_after();
        const uint32_t sa = smem0 + s * STAGE_BYTES;
#pragma unroll
        for (int k = 0; k < DWT_BK / TC_UMMA_K; ++k) {
          const uint32_t koff = k * TC_UMMA_K * 128;           // 8 node rows of 128 B
          const uint64_t da = make_desc_mn_sw128_32b(sa + koff, DWT_BK * 128);
          const uint64_t db = make_desc_mn_sw128_32b(sa + NA * DWT_A_BYTES + koff, DWT_BK * 128);
          tc_mma_tf32(tmem_base, da, db, idesc, (kb | k) ? 1u : 0u);
          if (NA == 2) {
            const uint64_t dl = make_desc_mn_sw128_32b(sa + DWT_A_BYTES + koff, DWT_BK * 128);
            tc_mma_tf32(tmem_base, dl, db, idesc, 1u);
          }
          if (XS) {                                            // T_hi^T X_lo
            const uint64_t dxl = make_desc_mn_sw128_32b(sa + NA * DWT_A_BYTES + DWT_B_BYTES + koff, DWT_BK * 128);
            tc_mma_tf32(tmem_base, da, dxl, idesc, 1u);
          }
        }
        tc_commit(smem_u32(&bar_empty[s]));
        if (kb == num_kb - 1) tc_commit(smem_u32(&bar_tmem_full));
        if (++s == STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (XS && warp >= 8) {   // ===== converters: X tile -> X_hi (in place) | X_lo =====
    const int cw = warp - 8;
    int s = 0;
    uint32_t ph = 0;
    for (int kb = 0; kb < num_kb; ++kb) {
      mbar_wait(smem_u32(&bar_full[s]), ph);
      const uint32_t sx = smem0 + s * STAGE_BYTES + NA * DWT_A_BYTES;
      split_tile_hi_lo(sx, sx + DWT_B_BYTES, DWT_B_BYTES, cw, lane);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&bar_conv[s]));
      if (++s == STAGES) { s = 0; ph ^= 1; }
    }
  } else if (warp >= 4 && warp < 8) {
    dw_epilogue(p, tmem_base, smem_u32(&bar_tmem_full), num_kb, col0, warp & 3, lane);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem_base));
  }
}

// [rows, cols] fp32 row-major, box = 32 cols x 32 rows, SWIZZLE_128B with 32 B atoms (MN-major tf32)
static int make_map_mn(CUtensorMap* m, const float* base, int64_t rows, int64_t cols, int64_t ld) {
  const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t gstr[1] = {(cuuint64_t)ld * 4};
  const cuuint32_t box[2] = {32, (cuuint32_t)DWT_BK};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = encode_fn()(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim, gstr, box,
                                 estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B,
                                 CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("dw_tc: cuTensorMapEncodeTiled failed (%d)", (int)r);
    return 2;
  }
  return 0;
}

// node splits of the dW GEMMs for N > 0: one wave of (column tile x split) CTAs, at least four stages of DWT_BK rows per
// split; *rps = rows per split (a multiple of DWT_BK)
static int dw_node_splits(int64_t N, int tiles, int64_t* rps) {
  int nsplit = num_sms() / tiles;
  const int64_t max_split = ceil_div(N, 4 * DWT_BK);
  if (nsplit > max_split) nsplit = (int)max_split;
  if (nsplit < 1) nsplit = 1;
  *rps = ceil_div(ceil_div(N, nsplit), DWT_BK) * DWT_BK;
  return (int)ceil_div(N, *rps);
}

__global__ void k_split_rows_hi_lo(const float* __restrict__ t, int64_t n, float* __restrict__ hi,
                                   float* __restrict__ lo) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float v = t[i];
    const float h = __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
    hi[i] = h;
    lo[i] = __uint_as_float((__float_as_uint(v - h) + 0x1000u) & 0xFFFFE000u);   // round to nearest: no sign bias
  }
}

// t: [N, n_out] (row pitch ldt == n_out).  hi_scratch / lo_scratch: N * n_out floats each (TF32X3 only).
int dw_tc(const float* x, int64_t N, int64_t K, const float* t, int64_t ldt, int n_out, float* hi_scratch,
          float* lo_scratch, float* partial, float* dw_a, int64_t ldw_a, int64_t k0_a, float* dw_b, int64_t ldw_b, int64_t k0_b,
          int mode, cudaStream_t st) {
  BIGCN_CHECK_ARG(encode_fn() != nullptr, "dw_tc: cuTensorMapEncodeTiled is unavailable in this driver");
  BIGCN_CHECK_ARG(K % 4 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0, "dw_tc: x must be TMA-addressable");
  BIGCN_CHECK_ARG(ldt == n_out && (n_out == 64 || n_out == 128), "dw_tc: t must be dense [N, 64|128]");
  if (K == 0) return 0;
  if (mode == BIGCN_GEMM_BF16)
    return dw_bf16(x, N, K, t, n_out, hi_scratch, lo_scratch, partial, dw_a, ldw_a, k0_a, dw_b, ldw_b, k0_b, st);
  const int na = mode == BIGCN_GEMM_TF32 ? 1 : 2;   // TF32X2, TF32X3 and MIXED split T
  const bool xsplit = mode == BIGCN_GEMM_TF32X3;    // ... and TF32X3 splits X in shared memory as well
  const int tiles = (int)ceil_div(K, DWT_N);
  int nsplit = 1;
  if (N == 0) {
    cudaMemsetAsync(partial, 0, (size_t)K * n_out * sizeof(float), st);
  } else {
    int64_t rps = 0;
    nsplit = dw_node_splits(N, tiles, &rps);
    const float* t_hi = t;
    const float* t_lo = t;
    if (na == 2) {
      BIGCN_CHECK_ARG(hi_scratch != nullptr && lo_scratch != nullptr, "dw_tc: TF32X3 needs the split scratch");
      float* hi = hi_scratch;
      float* lo = lo_scratch;
      k_split_rows_hi_lo<<<num_sms() * 4, 256, 0, st>>>(t, N * n_out, hi, lo);
      BIGCN_CHECK_LAUNCH("k_split_rows_hi_lo");
      t_hi = hi;
      t_lo = lo;
    }
    CUtensorMap mx, mt, ml;
    if (int rc = make_map_mn(&mx, x, N, K, K)) return rc;
    if (int rc = make_map_mn(&mt, t_hi, N, n_out, n_out)) return rc;
    if (int rc = make_map_mn(&ml, t_lo, N, n_out, n_out)) return rc;
    DwtParams p;
    p.partial = partial; p.N = N; p.K = K; p.n_out = n_out; p.rows_per_split = (int)rps;
    const int stages = xsplit ? 2 : (na == 1 ? 4 : 3);
    const size_t smem = (size_t)stages * (na * DWT_A_BYTES + (xsplit ? 2 : 1) * DWT_B_BYTES) + 1024;
    static bool attr = false;
    if (!attr) {
      cudaFuncSetAttribute(k_dw_tc<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * (DWT_A_BYTES + DWT_B_BYTES) + 1024);
      cudaFuncSetAttribute(k_dw_tc<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 3 * (2 * DWT_A_BYTES + DWT_B_BYTES) + 1024);
      cudaFuncSetAttribute(k_dw_tc<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * (2 * DWT_A_BYTES + 2 * DWT_B_BYTES) + 1024);
      attr = true;
    }
    if (na == 1) k_dw_tc<1, false><<<dim3(tiles, nsplit), TC_THREADS, smem, st>>>(mx, mt, ml, p);
    else if (!xsplit) k_dw_tc<2, false><<<dim3(tiles, nsplit), TC_THREADS, smem, st>>>(mx, mt, ml, p);
    else k_dw_tc<2, true><<<dim3(tiles, nsplit), TC_THREADS_XS, smem, st>>>(mx, mt, ml, p);
    BIGCN_CHECK_LAUNCH("k_dw_tc");
  }
  return dw_reduce_launch(partial, nsplit, K, n_out, dw_a, ldw_a, k0_a, dw_b, ldw_b, k0_b, st);
}


// =====================================================================================
// BIGCN_GEMM_BF16: x arrives as bf16 and is read from HBM as it is (half the bytes of fp32).  A bf16 x is exact, so the
// only rounding left is in the small operand (W forward, T backward): it is split into NT bf16 terms
//   t0 = bf16(v), t1 = bf16(v - t0), t2 = bf16(v - t0 - t1)
// (each difference exact in fp32) and every term takes one kind::f16 MMA against the same x tile into one fp32 TMEM
// accumulator.  Three terms carry 24 significant bits, as many as fp32; two carry 16 and fail the fp64 bars (DESIGN.md
// section 8 has the measurements behind the term count).
template <int NT>
__device__ __forceinline__ void bf16_terms(float v, __nv_bfloat16 (&t)[NT]) {
  float r = v;
#pragma unroll
  for (int i = 0; i < NT; ++i) {
    t[i] = __float2bfloat16_rn(r);
    r -= __bfloat162float(t[i]);
  }
}
constexpr int BF_NT = 3;   // bf16 terms of the small operand

// terms of the [64, K] weight w (row pitch ldw) of direction d: out[t][d * 64 + r][k], [NT][n_out][K] bf16
template <int NT>
__global__ void k_split_w_bf16(const float* __restrict__ w, int64_t ldw, int64_t K, int n_out, int d,
                               __nv_bfloat16* __restrict__ out) {
  const int64_t n = 64 * K;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / K, k = i % K;
    __nv_bfloat16 t[NT];
    bf16_terms<NT>(w[r * ldw + k], t);
#pragma unroll
    for (int j = 0; j < NT; ++j) out[((int64_t)j * n_out + d * 64 + r) * K + k] = t[j];
  }
}

// ---- forward  Y[N, n_out] = X[N, K] * W^T  with X bf16 -------------------------------------------------------------
// Same warp roles, 256-row tiles (two M = 128 accumulators sharing every B tile), split-K and epilogue as k_xw_tc.
// K blocks of 32 elements = one 64 B row of the SWIZZLE_64B layout: a stage is 16 KB of X plus NT x 8 KB of W terms
// (40 KB at NT = 3: five stages).  With 64-element blocks and the 128B swizzle a stage would be
// 80 KB and only two would fit.
constexpr int BF_BLOCK_K = 32;
constexpr int BF_UMMA_K = 16;
constexpr int BF_A_BYTES = TC_BLOCK_M * 64;   // 16 KB
constexpr int BF_B_BYTES = 128 * 64;          // 8 KB: one W term, up to 128 output rows
constexpr int BF_XW_STAGES = 5;
template <int NT>
constexpr int bf_xw_smem() { return BF_XW_STAGES * (BF_A_BYTES + NT * BF_B_BYTES) + 1024; }

template <int NT>
__global__ void __launch_bounds__(TC_THREADS, 1)
k_xw_bf16(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w, const TcParams p) {
  constexpr int STAGES = BF_XW_STAGES;
  constexpr int STAGE_BYTES = BF_A_BYTES + NT * BF_B_BYTES;
  extern __shared__ __align__(1024) uint8_t tc_smem[];
  __shared__ __align__(8) uint64_t bar_full[STAGES];
  __shared__ __align__(8) uint64_t bar_empty[STAGES];
  __shared__ __align__(8) uint64_t bar_tmem_full, bar_tmem_empty;
  __shared__ uint32_t tmem_base_s;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t smem0 = (smem_u32(tc_smem) + 1023u) & ~1023u;
  const int kb0 = blockIdx.y * p.kb_per, kb1 = min(p.num_kb, kb0 + p.kb_per);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_x);
    tma_prefetch_desc(&map_w);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(smem_u32(&bar_full[s]), 1);
      mbar_init(smem_u32(&bar_empty[s]), 1);
    }
    mbar_init(smem_u32(&bar_tmem_full), 1);
    mbar_init(smem_u32(&bar_tmem_empty), 4);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(smem_u32(&tmem_base_s)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp == 0) {
    if (lane == 0) {   // ===== TMA producer =====
      int s = 0;
      uint32_t ph = 0;
      const uint32_t tx = (uint32_t)(BF_A_BYTES + NT * p.n_out * 64);
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        const int m0 = tile * TC_BLOCK_M;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(smem_u32(&bar_empty[s]), ph ^ 1);
          const uint32_t full = smem_u32(&bar_full[s]);
          const uint32_t sa = smem0 + s * STAGE_BYTES;
          mbar_expect_tx(full, tx);
          tma_load_2d(sa, &map_x, full, kb * BF_BLOCK_K, m0);
#pragma unroll
          for (int t = 0; t < NT; ++t) tma_load_2d(sa + BF_A_BYTES + t * BF_B_BYTES, &map_w, full, kb * BF_BLOCK_K, t * p.n_out);
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {   // ===== MMA issuer =====
      const uint32_t idesc = make_idesc_bf16(128, p.n_out);
      int s = 0;
      uint32_t ph = 0, tile_ph = 0;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, tile_ph ^= 1) {
        mbar_wait(smem_u32(&bar_tmem_empty), tile_ph ^ 1);
        tc_fence_after();
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(smem_u32(&bar_full[s]), ph);
          tc_fence_after();
          const uint32_t sa = smem0 + s * STAGE_BYTES;
#pragma unroll
          for (int k = 0; k < BF_BLOCK_K / BF_UMMA_K; ++k) {
            const uint32_t koff = k * BF_UMMA_K * 2;         // 32 B per K step inside the 64 B row
            const uint64_t da0 = make_desc_k_sw64(sa + koff);
            const uint64_t da1 = make_desc_k_sw64(sa + 128 * 64 + koff);
#pragma unroll
            for (int t = 0; t < NT; ++t) {
              const uint64_t db = make_desc_k_sw64(sa + BF_A_BYTES + t * BF_B_BYTES + koff);
              const uint32_t acc = ((kb - kb0) | k | t) ? 1u : 0u;
              tc_mma_f16(tmem_base, da0, db, idesc, acc);
              tc_mma_f16(tmem_base + 128, da1, db, idesc, acc);
            }
          }
          tc_commit(smem_u32(&bar_empty[s]));
          if (kb == kb1 - 1) tc_commit(smem_u32(&bar_tmem_full));
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp >= 4) {
    xw_epilogue(p, tmem_base, smem_u32(&bar_tmem_full), smem_u32(&bar_tmem_empty), warp & 3, lane);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem_base));
  }
}

// x: bf16 [N, K]; w[0], w[1]: fp32 [64, K] (row pitch ldw); scratch: at least 3 * n_out * K bf16 (the W terms)
static int xw_bf16(const void* x, int64_t N, int64_t K, const float* const* w, int64_t ldw, int n_out, float* scratch,
                   float* y, int64_t ldy, cudaStream_t st, float* partial) {
  if (N == 0) return 0;
  BIGCN_CHECK_ARG(x != nullptr, "xw (bf16): NULL x");
  BIGCN_CHECK_ARG(K % 8 == 0, "xw (bf16): in_feats must be a multiple of 8 for TMA (16 B rows), got %lld", (long long)K);
  BIGCN_CHECK_ARG((reinterpret_cast<uintptr_t>(x) & 15) == 0, "xw (bf16): x must be 16-byte aligned");
  BIGCN_CHECK_ARG(scratch != nullptr, "xw (bf16): needs the weight scratch");
  __nv_bfloat16* terms = reinterpret_cast<__nv_bfloat16*>(scratch);
  for (int d = 0; d < n_out / 64; ++d) {
    k_split_w_bf16<BF_NT><<<num_sms() * 2, 256, 0, st>>>(w[d], ldw, K, n_out, d, terms);
    BIGCN_CHECK_LAUNCH("k_split_w_bf16");
  }
  CUtensorMap mx, mw;
  if (int rc = make_map_bf16(&mx, x, N, K, K, BF_BLOCK_K, TC_BLOCK_M, CU_TENSOR_MAP_SWIZZLE_64B)) return rc;
  if (int rc = make_map_bf16(&mw, terms, (int64_t)BF_NT * n_out, K, K, BF_BLOCK_K, n_out, CU_TENSOR_MAP_SWIZZLE_64B)) return rc;
  TcParams p;
  p.y = y; p.ldy = ldy; p.N = N; p.K = K; p.n_out = n_out;
  p.num_tiles = (int)ceil_div(N, TC_BLOCK_M);
  p.num_kb = (int)ceil_div(K, BF_BLOCK_K);
  const int grid_x = p.num_tiles < num_sms() ? p.num_tiles : num_sms();
  const int nsplit = xw_split_k(p, partial);
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(k_xw_bf16<BF_NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, bf_xw_smem<BF_NT>());
    attr = true;
  }
  const dim3 grid(grid_x, nsplit);
  k_xw_bf16<BF_NT><<<grid, TC_THREADS, bf_xw_smem<BF_NT>(), st>>>(mx, mw, p);
  BIGCN_CHECK_LAUNCH("k_xw_bf16");
  if (nsplit > 1) {
    int rb = (int)ceil_div(N * (n_out / 4), 256);
    if (rb > num_sms() * 4) rb = num_sms() * 4;
    k_xw_splitk_reduce<<<rb, 256, 0, st>>>(partial, nsplit, N, n_out, y, ldy);
    BIGCN_CHECK_LAUNCH("k_xw_splitk_reduce");
  }
  return 0;
}

// ---- weight gradient  dW^T[k, o] = sum_i X[i, k] * T[i, o]  with X bf16 -------------------------------------------
// As k_dw_tc (D[128 outputs, 256 columns of X] over the node axis, one wave of (column tile x node split) CTAs, ordered
// split-K reduce), with 16-bit MN-major operands: SWIZZLE_128B atoms of 64 elements x 8 node rows, TMA boxes of
// 64 columns x 32 node rows.  A stage is 32 node rows (two K = 16 MMAs per term): NT x 8 KB of T terms + 16 KB of X.
constexpr int DWB_BK = 32;
constexpr int DWB_A_BYTES = 2 * DWB_BK * 128;   // one T term: 128 outputs = 2 blocks of 64
constexpr int DWB_B_BYTES = 4 * DWB_BK * 128;   // 256 columns of X = 4 blocks of 64
constexpr int BF_DW_STAGES = 5;
template <int NT>
constexpr int bf_dw_smem() { return BF_DW_STAGES * (NT * DWB_A_BYTES + DWB_B_BYTES) + 1024; }
__host__ __device__ constexpr uint32_t make_idesc_bf16_mn(int m, int n) {
  return make_idesc_bf16(m, n) | (1u << 15) | (1u << 16);   // a_major = b_major = MN
}

template <int NT>
__global__ void __launch_bounds__(TC_THREADS, 1)
k_dw_bf16(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_t0,
          const __grid_constant__ CUtensorMap map_t1, const __grid_constant__ CUtensorMap map_t2, const DwtParams p) {
  static_assert(DWB_BK == DWT_BK, "dw_tc's node splits are multiples of DWT_BK");
  constexpr int STAGES = BF_DW_STAGES;
  constexpr int STAGE_BYTES = NT * DWB_A_BYTES + DWB_B_BYTES;   // [T0 | T1 | (T2) | X]
  extern __shared__ __align__(1024) uint8_t tc_smem[];
  __shared__ __align__(8) uint64_t bar_full[STAGES];
  __shared__ __align__(8) uint64_t bar_empty[STAGES];
  __shared__ __align__(8) uint64_t bar_tmem_full;
  __shared__ uint32_t tmem_base_s;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t smem0 = (smem_u32(tc_smem) + 1023u) & ~1023u;
  const int col0 = blockIdx.x * DWT_N;
  const int64_t r_begin = (int64_t)blockIdx.y * p.rows_per_split;
  const int64_t r_end = min(p.N, r_begin + p.rows_per_split);
  const int num_kb = r_end > r_begin ? (int)((r_end - r_begin + DWB_BK - 1) / DWB_BK) : 0;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_x);
    tma_prefetch_desc(&map_t0);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(smem_u32(&bar_full[s]), 1);
      mbar_init(smem_u32(&bar_empty[s]), 1);
    }
    mbar_init(smem_u32(&bar_tmem_full), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(smem_u32(&tmem_base_s)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp == 0) {
    if (lane == 0) {   // ===== TMA producer =====
      int s = 0;
      uint32_t ph = 0;
      // both 64-output blocks of every term are always loaded: a block beyond n_out is out of bounds -> zero filled
      const uint32_t tx = (uint32_t)(NT * DWB_A_BYTES + DWB_B_BYTES);
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(smem_u32(&bar_empty[s]), ph ^ 1);
        const uint32_t full = smem_u32(&bar_full[s]);
        const uint32_t sa = smem0 + s * STAGE_BYTES;
        const int row = (int)(r_begin + (int64_t)kb * DWB_BK);
        mbar_expect_tx(full, tx);
#pragma unroll
        for (int mb = 0; mb < 2; ++mb) {
          tma_load_2d(sa + mb * (DWB_BK * 128), &map_t0, full, mb * 64, row);
          tma_load_2d(sa + DWB_A_BYTES + mb * (DWB_BK * 128), &map_t1, full, mb * 64, row);
          if (NT == 3) tma_load_2d(sa + 2 * DWB_A_BYTES + mb * (DWB_BK * 128), &map_t2, full, mb * 64, row);
        }
#pragma unroll
        for (int nb = 0; nb < 4; ++nb)
          tma_load_2d(sa + NT * DWB_A_BYTES + nb * (DWB_BK * 128), &map_x, full, col0 + nb * 64, row);
        if (++s == STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {   // ===== MMA issuer =====
      const uint32_t idesc = make_idesc_bf16_mn(128, DWT_N);
      int s = 0;
      uint32_t ph = 0;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(smem_u32(&bar_full[s]), ph);
        tc_fence_after();
        const uint32_t sa = smem0 + s * STAGE_BYTES;
#pragma unroll
        for (int k = 0; k < DWB_BK / BF_UMMA_K; ++k) {
          const uint32_t koff = k * BF_UMMA_K * 128;           // 16 node rows of 128 B
          const uint64_t db = make_desc_mn_sw128_16b(sa + NT * DWB_A_BYTES + koff, DWB_BK * 128);
#pragma unroll
          for (int t = 0; t < NT; ++t) {
            const uint64_t da = make_desc_mn_sw128_16b(sa + t * DWB_A_BYTES + koff, DWB_BK * 128);
            tc_mma_f16(tmem_base, da, db, idesc, (kb | k | t) ? 1u : 0u);
          }
        }
        tc_commit(smem_u32(&bar_empty[s]));
        if (kb == num_kb - 1) tc_commit(smem_u32(&bar_tmem_full));
        if (++s == STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp >= 4) {
    dw_epilogue(p, tmem_base, smem_u32(&bar_tmem_full), num_kb, col0, warp & 3, lane);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem_base));
  }
}

// terms of t [n elements]: t0 -> t01[i], t1 -> t01[n + i], t2 -> t2[i]
template <int NT>
__global__ void k_split_rows_bf16(const float* __restrict__ t, int64_t n, __nv_bfloat16* __restrict__ t01,
                                  __nv_bfloat16* __restrict__ t2) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    __nv_bfloat16 v[NT];
    bf16_terms<NT>(t[i], v);
    t01[i] = v[0];
    t01[n + i] = v[1];
    if (NT == 3) t2[i] = v[NT - 1];
  }
}

// x: bf16 [N, K]; t: fp32 [N, n_out]; scratch01: N * n_out floats (terms 0 and 1 as bf16), scratch2: N * n_out floats
static int dw_bf16(const void* x, int64_t N, int64_t K, const float* t, int n_out, float* scratch01, float* scratch2,
                   float* partial, float* dw_a, int64_t ldw_a, int64_t k0_a, float* dw_b, int64_t ldw_b, int64_t k0_b,
                   cudaStream_t st) {
  BIGCN_CHECK_ARG(N == 0 || (x != nullptr && K % 8 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0),
                  "dw (bf16): x must be 16-byte aligned with in_feats a multiple of 8 (TMA)");
  BIGCN_CHECK_ARG(scratch01 != nullptr && scratch2 != nullptr, "dw (bf16): needs the split scratch");
  const int tiles = (int)ceil_div(K, DWT_N);
  int nsplit = 1;
  if (N == 0) {
    cudaMemsetAsync(partial, 0, (size_t)K * n_out * sizeof(float), st);
  } else {
    int64_t rps = 0;
    nsplit = dw_node_splits(N, tiles, &rps);
    __nv_bfloat16* t01 = reinterpret_cast<__nv_bfloat16*>(scratch01);
    __nv_bfloat16* t2 = reinterpret_cast<__nv_bfloat16*>(scratch2);
    k_split_rows_bf16<BF_NT><<<num_sms() * 4, 256, 0, st>>>(t, N * n_out, t01, t2);
    BIGCN_CHECK_LAUNCH("k_split_rows_bf16");
    CUtensorMap mx, m0, m1, m2;
    if (int rc = make_map_bf16(&mx, x, N, K, K, 64, DWB_BK, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    if (int rc = make_map_bf16(&m0, t01, N, n_out, n_out, 64, DWB_BK, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    if (int rc = make_map_bf16(&m1, t01 + N * n_out, N, n_out, n_out, 64, DWB_BK, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    if (int rc = make_map_bf16(&m2, t2, N, n_out, n_out, 64, DWB_BK, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    DwtParams p;
    p.partial = partial; p.N = N; p.K = K; p.n_out = n_out; p.rows_per_split = (int)rps;
    static bool attr = false;
    if (!attr) {
      cudaFuncSetAttribute(k_dw_bf16<BF_NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, bf_dw_smem<BF_NT>());
      attr = true;
    }
    k_dw_bf16<BF_NT><<<dim3(tiles, nsplit), TC_THREADS, bf_dw_smem<BF_NT>(), st>>>(mx, m0, m1, m2, p);
    BIGCN_CHECK_LAUNCH("k_dw_bf16");
  }
  return dw_reduce_launch(partial, nsplit, K, n_out, dw_a, ldw_a, k0_a, dw_b, ldw_b, k0_b, st);
}


// =====================================================================================
// Input gradient  dX[N, K] = T[N, 64 n_w] * Wcat[64 n_w, K],  Wcat = [W_0; W_1] the [64, K] conv1.lin weights
// (SURVEY appendix B: dX = T1 W1, summed over the directions by the reduction itself).
// D[M = 128 rows of T, N = 256 columns of dX] with a reduction depth of only 64 n_w: both operands are small (T is
// 16 MB, W 2.5 MB at Twitter scale) and the [N, K] output dominates the bytes.  3xTF32, T_hi W_hi + T_hi W_lo +
// T_lo W_hi: both operands are split beforehand (k_split_rows_hi_lo, k_split_wT_hi_lo), so the MMA loop has no
// converter warps.  W is laid out transposed as [K][64 n_w] (the forward's w1T layout): the B operand is K-major with
// a 256 / 512 B row pitch that TMA can address whatever K is; rows >= K and >= N are zero-filled by TMA and the
// column tail is cut in the epilogue.  Persistent CTAs walk the (row tile, column tile) pairs; the accumulator is
// double-buffered in TMEM (2 x 256 columns), so eight epilogue warps drain tile i while the MMAs of tile i + 1 run.
//   warp 0 : TMA producer      warp 1 : MMA issuer      warp 2 : TMEM allocator      warps 4-11 : epilogue
// Every output element is written once by one thread from one accumulator: deterministic, no atomics.
constexpr int DX_BM = 128;
constexpr int DX_BN = 256;
constexpr int DX_A_BYTES = DX_BM * 128;                             // 16 KB: 128 rows x 32 fp32
constexpr int DX_B_BYTES = DX_BN * 128;                             // 32 KB: 256 rows x 32 fp32
constexpr int DX_STAGE_BYTES = 2 * DX_A_BYTES + 2 * DX_B_BYTES;     // [T_hi | T_lo | W_hi | W_lo] = 96 KB
constexpr int DX_STAGES = 2;
constexpr int DX_THREADS = 384;
constexpr int DX_SMEM = DX_STAGES * DX_STAGE_BYTES + 1024;

struct DxParams {
  void* dx;          // [N][K] fp32 or bf16
  int64_t N, K;
  int num_kb;        // 64 n_w / 32
  int col_tiles;     // ceil(K / 256)
  int num_tiles;     // ceil(N / 128) * col_tiles
  int vec;           // 1: dx rows can take 16 B stores (K a multiple of 16 B, dx 16 B aligned)
};

// one thread's 32 consecutive accumulator columns of one row -> dx (fp32, or bf16 rounded to nearest even once)
template <typename OutT>
__device__ __forceinline__ void dx_store32(const DxParams& p, int64_t row, int64_t col, const uint32_t (&r)[32]) {
  if (row >= p.N || col >= p.K) return;
  OutT* dst = reinterpret_cast<OutT*>(p.dx) + row * p.K + col;
  if (p.vec && col + 32 <= p.K) {
    if constexpr (sizeof(OutT) == 4) {
      float4* d4 = reinterpret_cast<float4*>(dst);
#pragma unroll
      for (int j = 0; j < 8; ++j)
        d4[j] = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]), __uint_as_float(r[4 * j + 2]),
                            __uint_as_float(r[4 * j + 3]));
    } else {
      uint32_t h[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const __nv_bfloat162 b = __floats2bfloat162_rn(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1]));
        h[j] = *reinterpret_cast<const uint32_t*>(&b);
      }
      uint4* d4 = reinterpret_cast<uint4*>(dst);
#pragma unroll
      for (int j = 0; j < 4; ++j) d4[j] = make_uint4(h[4 * j], h[4 * j + 1], h[4 * j + 2], h[4 * j + 3]);
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      if (col + j < p.K) {
        if constexpr (sizeof(OutT) == 4) dst[j] = __uint_as_float(r[j]);
        else dst[j] = __float2bfloat16_rn(__uint_as_float(r[j]));
      }
    }
  }
}

template <typename OutT>
__global__ void __launch_bounds__(DX_THREADS, 1)
k_dx_tc(const __grid_constant__ CUtensorMap map_t, const __grid_constant__ CUtensorMap map_tlo,
        const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_wlo, const DxParams p) {
  extern __shared__ __align__(1024) uint8_t tc_smem[];
  __shared__ __align__(8) uint64_t bar_full[DX_STAGES];
  __shared__ __align__(8) uint64_t bar_empty[DX_STAGES];
  __shared__ __align__(8) uint64_t bar_tmem_full[2];
  __shared__ __align__(8) uint64_t bar_tmem_empty[2];
  __shared__ uint32_t tmem_base_s;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t smem0 = (smem_u32(tc_smem) + 1023u) & ~1023u;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_t);
    tma_prefetch_desc(&map_tlo);
    tma_prefetch_desc(&map_w);
    tma_prefetch_desc(&map_wlo);
    for (int s = 0; s < DX_STAGES; ++s) {
      mbar_init(smem_u32(&bar_full[s]), 1);
      mbar_init(smem_u32(&bar_empty[s]), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(smem_u32(&bar_tmem_full[a]), 1);
      mbar_init(smem_u32(&bar_tmem_empty[a]), 8);   // the eight epilogue warps
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {   // 512 TMEM columns: two 128 x 256 fp32 accumulators
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&tmem_base_s)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp == 0) {
    if (lane == 0) {   // ===== TMA producer =====
      int s = 0;
      uint32_t ph = 0;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        const int m0 = (tile / p.col_tiles) * DX_BM;
        const int c0 = (tile % p.col_tiles) * DX_BN;
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(smem_u32(&bar_empty[s]), ph ^ 1);
          const uint32_t full = smem_u32(&bar_full[s]);
          const uint32_t sa = smem0 + s * DX_STAGE_BYTES;
          mbar_expect_tx(full, (uint32_t)DX_STAGE_BYTES);
          tma_load_2d(sa, &map_t, full, kb * 32, m0);
          tma_load_2d(sa + DX_A_BYTES, &map_tlo, full, kb * 32, m0);
          tma_load_2d(sa + 2 * DX_A_BYTES, &map_w, full, kb * 32, c0);
          tma_load_2d(sa + 2 * DX_A_BYTES + DX_B_BYTES, &map_wlo, full, kb * 32, c0);
          if (++s == DX_STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {   // ===== MMA issuer =====
      const uint32_t idesc = make_idesc_tf32(DX_BM, DX_BN);
      int s = 0;
      uint32_t ph = 0;
      int it = 0;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
        const int a = it & 1;
        mbar_wait(smem_u32(&bar_tmem_empty[a]), ((it >> 1) & 1) ^ 1);   // the epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t d = tmem_base + (uint32_t)(a * DX_BN);
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(smem_u32(&bar_full[s]), ph);
          tc_fence_after();
          const uint32_t sa = smem0 + s * DX_STAGE_BYTES;
#pragma unroll
          for (int k = 0; k < 32 / TC_UMMA_K; ++k) {
            const uint32_t koff = k * TC_UMMA_K * 4;
            const uint64_t dt = make_desc_k_sw128(sa + koff);
            const uint64_t dtl = make_desc_k_sw128(sa + DX_A_BYTES + koff);
            const uint64_t dw = make_desc_k_sw128(sa + 2 * DX_A_BYTES + koff);
            const uint64_t dwl = make_desc_k_sw128(sa + 2 * DX_A_BYTES + DX_B_BYTES + koff);
            tc_mma_tf32(d, dt, dw, idesc, (kb | k) ? 1u : 0u);
            tc_mma_tf32(d, dt, dwl, idesc, 1u);
            tc_mma_tf32(d, dtl, dw, idesc, 1u);
          }
          tc_commit(smem_u32(&bar_empty[s]));
          if (kb == p.num_kb - 1) tc_commit(smem_u32(&bar_tmem_full[a]));
          if (++s == DX_STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp >= 4) {   // ===== epilogue: warp w reads TMEM lanes 32 (w % 4).. and one half of the 256 columns
    const int q = warp & 3, half = (warp - 4) >> 2;
    int it = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      const int a = it & 1;
      mbar_wait(smem_u32(&bar_tmem_full[a]), (it >> 1) & 1);
      tc_fence_after();
      const int64_t row = (int64_t)(tile / p.col_tiles) * DX_BM + q * 32 + lane;
      const int64_t col = (int64_t)(tile % p.col_tiles) * DX_BN + half * 128;
#pragma unroll 1
      for (int c = 0; c < 128; c += 32) {
        uint32_t r[32];
        tc_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(a * DX_BN + half * 128 + c), r);
        tc_wait_ld();
        dx_store32<OutT>(p, row, col + c, r);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&bar_tmem_empty[a]));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base));
  }
}

// Transposed hi / lo split of one direction's [64, K] weight into columns col0..col0+63 of [K][ldo]
__global__ void k_split_wT_hi_lo(const float* __restrict__ w, int64_t ldw, int64_t K, int ldo, int col0,
                                 float* __restrict__ hi, float* __restrict__ lo) {
  const int64_t n = 64 * K;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t k = i >> 6, r = i & 63;
    const float v = w[r * ldw + k];
    const float h = __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
    hi[k * ldo + col0 + r] = h;
    lo[k * ldo + col0 + r] = __uint_as_float((__float_as_uint(v - h) + 0x1000u) & 0xFFFFE000u);
  }
}

size_t dx_tc_scratch_floats(int64_t N, int64_t K, int n_w) {
  return (size_t)2 * H * n_w * (size_t)((N > 0 ? N : 1) + (K > 0 ? K : 1));
}

// t: [N, 64 n_w] dense; w[d]: [64, K] (row pitch ldw) for d < n_w; exactly one of dx (fp32) / dx_bf16 is set, [N, K]
// dense; scratch: dx_tc_scratch_floats(N, K, n_w) floats, 16 B aligned
int dx_tc(const float* t, int n_w, const float* const* w, int64_t ldw, int64_t N, int64_t K, float* dx, void* dx_bf16,
          float* scratch, cudaStream_t st) {
  BIGCN_CHECK_ARG(encode_fn() != nullptr, "x_dgrad: cuTensorMapEncodeTiled is unavailable in this driver");
  BIGCN_CHECK_ARG(n_w == 1 || n_w == 2, "x_dgrad: n_w must be 1 or 2");
  BIGCN_CHECK_ARG((dx != nullptr) != (dx_bf16 != nullptr), "x_dgrad: pass exactly one of dx / dx_bf16");
  BIGCN_CHECK_ARG(N >= 0 && K >= 0 && ldw >= K, "x_dgrad: bad sizes");
  if (N == 0 || K == 0) return 0;
  BIGCN_CHECK_ARG(t != nullptr && w[0] != nullptr && (n_w == 1 || w[1] != nullptr) && scratch != nullptr,
                  "x_dgrad: NULL argument");
  BIGCN_CHECK_ARG((reinterpret_cast<uintptr_t>(t) & 15) == 0 && (reinterpret_cast<uintptr_t>(scratch) & 15) == 0,
                  "x_dgrad: t and scratch must be 16-byte aligned");
  const int nk = H * n_w;
  float* t_hi = scratch;
  float* t_lo = t_hi + (size_t)N * nk;
  float* w_hi = t_lo + (size_t)N * nk;
  float* w_lo = w_hi + (size_t)K * nk;
  k_split_rows_hi_lo<<<num_sms() * 4, 256, 0, st>>>(t, N * nk, t_hi, t_lo);
  BIGCN_CHECK_LAUNCH("k_split_rows_hi_lo");
  for (int d = 0; d < n_w; ++d) {
    k_split_wT_hi_lo<<<num_sms() * 2, 256, 0, st>>>(w[d], ldw, K, nk, d * H, w_hi, w_lo);
    BIGCN_CHECK_LAUNCH("k_split_wT_hi_lo");
  }
  CUtensorMap mt, mtl, mw, mwl;
  if (int rc = make_map(&mt, t_hi, N, nk, nk, DX_BM)) return rc;
  if (int rc = make_map(&mtl, t_lo, N, nk, nk, DX_BM)) return rc;
  if (int rc = make_map(&mw, w_hi, K, nk, nk, DX_BN)) return rc;
  if (int rc = make_map(&mwl, w_lo, K, nk, nk, DX_BN)) return rc;
  const bool bf = dx_bf16 != nullptr;
  DxParams p;
  p.dx = bf ? dx_bf16 : static_cast<void*>(dx);
  p.N = N; p.K = K;
  p.num_kb = nk / 32;
  p.col_tiles = (int)ceil_div(K, DX_BN);
  p.num_tiles = (int)(ceil_div(N, DX_BM) * p.col_tiles);
  BIGCN_CHECK_ARG(ceil_div(N, DX_BM) * p.col_tiles < (int64_t)1 << 31, "x_dgrad: too many tiles");
  p.vec = (K % (bf ? 8 : 4) == 0) && (reinterpret_cast<uintptr_t>(p.dx) & 15) == 0;
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(k_dx_tc<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, DX_SMEM);
    cudaFuncSetAttribute(k_dx_tc<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, DX_SMEM);
    attr = true;
  }
  const int grid = p.num_tiles < num_sms() ? p.num_tiles : num_sms();
  if (bf) k_dx_tc<__nv_bfloat16><<<grid, DX_THREADS, DX_SMEM, st>>>(mt, mtl, mw, mwl, p);
  else k_dx_tc<float><<<grid, DX_THREADS, DX_SMEM, st>>>(mt, mtl, mw, mwl, p);
  BIGCN_CHECK_LAUNCH("k_dx_tc");
  return 0;
}

}  // namespace bigcn
