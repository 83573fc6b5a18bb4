// X * W^T and its weight-gradient X^T * T, exact-fp32 streaming path.
//
// Replaces GCNConv.lin (cuBLAS SGEMM) at BiGCN_Twitter.py:42,92 and the autograd
// transpose of it (dW1 = T1^T X, SURVEY.md appendix B).  X is the 5000-wide
// bag-of-words matrix (~99.7 % zeros, small integer counts): both kernels are pure
// HBM streams over X -- every 32 B sector of X is read exactly once -- that do
// FFMA work only for the non-zero entries they meet, in a fixed order (no atomics),
// so results are exact fp32 sums and bit-reproducible.  Dense inputs stay correct
// (every entry then takes the FFMA branch); the tcgen05 kind::tf32 GEMM in
// gemm_tc.cu is the path for those.
#include "kernels.cuh"

namespace bigcn {

// ------------------------------------------------------------------ y = x * wt
// warp per row; lane loads float4 strips of the row (512 B per warp-load, XW_U loads
// in flight), ballots the non-zeros and accumulates val * wt[k, :] (n_out floats,
// L1/L2 resident) into n_out/32 registers per lane.
constexpr int XW_U = 8;

// CAPTURE: lane 0 also records every non-zero (column, value) in the row's ELL slots and the
// exact count (xsparse.cu turns that into the CSR / CSC the sparse weight gradient sweeps).
// PRODUCT = false: capture only (bigcn_batch_prepare: the weights of the step that will use the batch do not exist yet).
template <int NOUT, bool VEC4, bool CAPTURE, bool PRODUCT = true>
__global__ void __launch_bounds__(256, 1) k_xw_scan(const float* __restrict__ x, int64_t N, int64_t K,
                                              const float* __restrict__ wt,
                                              float* __restrict__ y, int64_t ldy,
                                              int32_t* __restrict__ xs_cnt, int32_t* __restrict__ xs_col,
                                              float* __restrict__ xs_val) {
  constexpr int V = NOUT / 32;
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarp = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const uint64_t pol = l2_evict_first_policy();
  for (int64_t row = warp0; row < N; row += nwarp) {
    const float* xr = x + row * K;
    float acc[V];
#pragma unroll
    for (int j = 0; j < V; ++j) acc[j] = 0.f;
    int nz = 0;
    for (int64_t k0 = 0; k0 < K; k0 += 128 * XW_U) {
      float4 v[XW_U];
#pragma unroll
      for (int u = 0; u < XW_U; ++u) {
        const int64_t kk = k0 + u * 128 + lane * 4;
        if (VEC4) {
          v[u] = kk < K ? ldg_stream_f4_ef(xr + kk, pol) : make_float4(0.f, 0.f, 0.f, 0.f);
        } else {
          v[u].x = kk + 0 < K ? __ldg(xr + kk + 0) : 0.f;
          v[u].y = kk + 1 < K ? __ldg(xr + kk + 1) : 0.f;
          v[u].z = kk + 2 < K ? __ldg(xr + kk + 2) : 0.f;
          v[u].w = kk + 3 < K ? __ldg(xr + kk + 3) : 0.f;
        }
      }
#pragma unroll
      for (int u = 0; u < XW_U; ++u) {
        const bool any = (v[u].x != 0.f) | (v[u].y != 0.f) | (v[u].z != 0.f) | (v[u].w != 0.f);
        if (__ballot_sync(FULL_MASK, any) == 0u) continue;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const float comp = c == 0 ? v[u].x : (c == 1 ? v[u].y : (c == 2 ? v[u].z : v[u].w));
          unsigned m = __ballot_sync(FULL_MASK, comp != 0.f);
          while (m) {
            const int sl = __ffs(m) - 1;
            m &= m - 1;
            const float val = __shfl_sync(FULL_MASK, comp, sl);
            const int64_t k = k0 + u * 128 + sl * 4 + c;
            if (CAPTURE) {
              if (lane == 0 && nz < XS_ELL) {
                xs_col[row * XS_ELL + nz] = (int32_t)k;
                xs_val[row * XS_ELL + nz] = val;
              }
              ++nz;
            }
            if (!PRODUCT) continue;
            const float* wr = wt + k * NOUT + lane * V;
            if (V == 4) {
              const float4 w = *reinterpret_cast<const float4*>(wr);
              fma2(acc[0], acc[1], val, w.x, w.y);
              fma2(acc[2], acc[3], val, w.z, w.w);
            } else {
              const float2 w = *reinterpret_cast<const float2*>(wr);
              fma2(acc[0], acc[1], val, w.x, w.y);
            }
          }
        }
      }
    }
    if (PRODUCT) {
      float* yr = y + row * ldy + lane * V;
      if (V == 4)
        *reinterpret_cast<float4*>(yr) = make_float4(acc[0], acc[1], acc[2], acc[3]);
      else
        *reinterpret_cast<float2*>(yr) = make_float2(acc[0], acc[1]);
    }
    if (CAPTURE && lane == 0) xs_cnt[row] = nz;
  }
}

template <bool CAPTURE>
static int xw_scan_launch(const float* x, int64_t N, int64_t K, const float* wt, int n_out, float* y, int64_t ldy,
                          int32_t* xs_cnt, int32_t* xs_col, float* xs_val, int ctas_per_sm, cudaStream_t st) {
  if (N == 0) return 0;
  const bool vec4 = (K % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  int blocks = (int)ceil_div(N, 8);
  const int cap = num_sms() * ctas_per_sm;
  if (blocks > cap) blocks = cap;
  if (n_out == 128) {
    if (vec4) k_xw_scan<128, true, CAPTURE><<<blocks, 256, 0, st>>>(x, N, K, wt, y, ldy, xs_cnt, xs_col, xs_val);
    else k_xw_scan<128, false, CAPTURE><<<blocks, 256, 0, st>>>(x, N, K, wt, y, ldy, xs_cnt, xs_col, xs_val);
  } else {
    if (vec4) k_xw_scan<64, true, CAPTURE><<<blocks, 256, 0, st>>>(x, N, K, wt, y, ldy, xs_cnt, xs_col, xs_val);
    else k_xw_scan<64, false, CAPTURE><<<blocks, 256, 0, st>>>(x, N, K, wt, y, ldy, xs_cnt, xs_col, xs_val);
  }
  BIGCN_CHECK_LAUNCH("k_xw_scan");
  return 0;
}

int xw_fp32(const float* x, int64_t N, int64_t K, const float* wt, int n_out, float* y, int64_t ldy,
            cudaStream_t st) {
  return xw_scan_launch<false>(x, N, K, wt, n_out, y, ldy, nullptr, nullptr, nullptr, 8, st);
}
// 6 CTAs per SM (the stream is HBM-bound with ~200 KB in flight per SM either way): leaves room
// for the short kernels of the side stream to run beside it
int xw_fp32_capture(const float* x, int64_t N, int64_t K, const float* wt, int n_out, float* y, int64_t ldy,
                    const XSparse& xs, cudaStream_t st) {
  return xw_scan_launch<true>(x, N, K, wt, n_out, y, ldy, xs.cnt, xs.ell_col, xs.ell_val, 6, st);
}

// ---- the background pass over x (bigcn_batch_prepare): capture only, fed by the TMA engine -----------------------------
// One small persistent CTA per SM, CAPW warps, one ROW each: lane 0 of a warp streams its row into the warp's ring in shared
// memory with cp.async.bulk (4 KB chunks = the 1024-column blocks of the fused scan, L2 evict-first); every lane owns 32
// consecutive floats of a chunk, builds a bit mask of its non-zeros, and two warp scans place them in the row's ELL slots in
// exactly the slot order of k_xw_scan (same ELL contents; tools/capture_check.py).  The point is the footprint: 4 warps x 3
// stages -- 128 threads, 50 registers, 48 KB of shared memory per SM and at most CAPW * CAPS * 4 KB in flight per
// SM -- so the pass runs the whole length of a step without taking slots or registers from the step's own latency-bound
// kernels (DESIGN.md section 4: the chain feels the footprint of the pass, not its HBM traffic).
constexpr int CAP_CHUNK = 1024;   // floats per chunk
template <int CAPW, int CAPS>
__global__ void __launch_bounds__(32 * CAPW) k_x_capture_tma(const float* __restrict__ x, int64_t N, int64_t K,
                                                             int32_t* __restrict__ xs_cnt, int32_t* __restrict__ xs_col,
                                                             float* __restrict__ xs_val) {
  extern __shared__ __align__(128) float cap_smem[];
  float (*buf)[CAPS][CAP_CHUNK] = reinterpret_cast<float (*)[CAPS][CAP_CHUNK]>(cap_smem);
  __shared__ __align__(8) uint64_t full[CAPW][CAPS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int w = 0; w < CAPW; ++w)
      for (int s = 0; s < CAPS; ++s) mbar_init(smem_u32(&full[w][s]), 1);
    mbar_init_fence();
  }
  __syncthreads();
  // every warp is its own producer: lane 0 keeps CAPS chunks of the warp's row stream in flight (the chunk sequence of
  // a warp runs over its rows: row r0, chunks 0..nchunk-1, then row r0 + stride, ...)
  const int nchunk = (int)((K + CAP_CHUNK - 1) / CAP_CHUNK);
  const int64_t stride = (int64_t)gridDim.x * CAPW;
  const int64_t row0 = (int64_t)blockIdx.x * CAPW + warp;
  const uint64_t pol = l2_evict_first_policy();
  int64_t prow = row0;   // producer cursor
  int pc = 0;
  auto issue = [&](int s) {
    if (prow >= N) return;
    const int nfl = (int)min((int64_t)CAP_CHUNK, K - (int64_t)pc * CAP_CHUNK);
    const uint32_t fb = smem_u32(&full[warp][s]);
    mbar_expect_tx(fb, (uint32_t)nfl * 4);
    bulk_g2s_hint(smem_u32(&buf[warp][s][0]), x + prow * K + (int64_t)pc * CAP_CHUNK, (uint32_t)nfl * 4, fb, pol);
    if (++pc == nchunk) { pc = 0; prow += stride; }
  };
  if (lane == 0)
    for (int s = 0; s < CAPS; ++s) issue(s);
  int s = 0;
  uint32_t ph = 0;
  for (int64_t row = row0; row < N; row += stride) {
    int nz = 0;
    for (int c = 0; c < nchunk; ++c) {
      const int nfl = (int)min((int64_t)CAP_CHUNK, K - (int64_t)c * CAP_CHUNK);
      mbar_wait(smem_u32(&full[warp][s]), ph);
      // lane l owns floats [32 l, 32 l + 32) of the chunk: eight 16-byte reads, rotated by the lane so that the eight
      // lanes of a quarter-warp hit eight different bank groups; one bit per non-zero
      const float* seg = &buf[warp][s][0] + lane * 32;
      unsigned mask = 0;
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int pu = (u + lane) & 7;
        const float4 v = *reinterpret_cast<const float4*>(seg + 4 * pu);
        const unsigned m4 = (v.x != 0.f ? 1u : 0u) | (v.y != 0.f ? 2u : 0u) | (v.z != 0.f ? 4u : 0u) | (v.w != 0.f ? 8u : 0u);
        mask |= m4 << (4 * pu);
      }
      const int valid = nfl - lane * 32;   // the last chunk of a row is short: what lies behind it is a previous chunk
      if (valid < 32) mask = valid <= 0 ? 0u : (mask & ((1u << valid) - 1u));
      if (__ballot_sync(FULL_MASK, mask != 0u)) {
        // The slots of a row follow the order of the fused scan (k_xw_scan: per block of 128 floats, component q of the
        // float4s first, then the lane), because the product sums in slot order and must not depend on which pass
        // captured the row.  Four lanes own one block of 128: lane l holds float4s 8 (l & 3) .. + 8 of block l >> 2.
        // Counts per component, one byte each (<= 8 per lane, <= 32 per block and component, <= 128 per block):
        unsigned cq = 0;
#pragma unroll
        for (int q = 0; q < 4; ++q) cq |= (unsigned)__popc(mask & (0x11111111u << q)) << (8 * q);
        unsigned gincl = cq;   // inclusive scan over the four lanes of the block
#pragma unroll
        for (int d = 1; d < 4; d <<= 1) {
          const unsigned t = __shfl_up_sync(FULL_MASK, gincl, d, 4);
          if ((lane & 3) >= d) gincl += t;
        }
        const unsigned gt = __shfl_sync(FULL_MASK, gincl, 3, 4);            // the block's counts per component
        const unsigned qbase = (gt << 8) + (gt << 16) + (gt << 24);         // byte q: entries of components < q (< 128)
        const int bt = (int)((gt & 0xff) + ((gt >> 8) & 0xff) + ((gt >> 16) & 0xff) + (gt >> 24));
        int binc = bt;         // inclusive scan of the block totals over the eight blocks (every lane of a block holds bt)
#pragma unroll
        for (int d = 4; d < 32; d <<= 1) {
          const int t = __shfl_up_sync(FULL_MASK, binc, d);
          if (lane >= d) binc += t;
        }
        const int base = nz + binc - bt;
        unsigned next = qbase + (gincl - cq);   // byte q: this lane's next slot of component q inside the block
        const int col0 = c * CAP_CHUNK + lane * 32;
        while (mask) {
          const int p = __ffs(mask) - 1;
          mask &= mask - 1;
          const int sh = 8 * (p & 3);
          const int slot = base + (int)((next >> sh) & 0xffu);
          next += 1u << sh;
          if (slot < XS_ELL) {
            xs_col[row * XS_ELL + slot] = col0 + p;
            xs_val[row * XS_ELL + slot] = seg[p];
          }
        }
        nz += __shfl_sync(FULL_MASK, binc, 31);
      }
      // the stage is read: hand it back to the TMA engine (generic-proxy reads before the async-proxy write)
      __syncwarp();
      if (lane == 0) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        issue(s);
      }
      if (++s == CAPS) { s = 0; ph ^= 1; }
    }
    if (lane == 0) xs_cnt[row] = nz;
  }
}

// The LDG form of the same pass (k_xw_scan<..., capture, no product>): launched as MANY SHORT CTAs (8 rows each, one per warp,
// ~160 KB of x) so that slots free up every few microseconds and the block scheduler hands them to the step's own
// (higher-priority) kernels first.  Used when x is not 16-byte addressable, and for the A/B (debug key 10 = 9:
// tools/stepbench.py, bench.py's unpaced capture entry).
int x_capture(const float* x, int64_t N, int64_t K, const XSparse& xs, cudaStream_t st) {
  if (N == 0) return 0;
  const bool vec4 = (K % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  if (vec4 && debug_knob(10) != 9) {   // TMA-fed persistent form
    constexpr int CAPW = 4, CAPS = 3, smem = CAPW * CAPS * CAP_CHUNK * 4;
    static bool attr = false;
    if (!attr) {
      cudaFuncSetAttribute(k_x_capture_tma<CAPW, CAPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
      attr = true;
    }
    const int grid = (int)min((int64_t)num_sms(), ceil_div(N, 4));
    k_x_capture_tma<CAPW, CAPS><<<grid, 32 * CAPW, smem, st>>>(x, N, K, xs.cnt, xs.ell_col, xs.ell_val);
    BIGCN_CHECK_LAUNCH("k_x_capture_tma");
    return 0;
  }
  const int blocks = (int)ceil_div(N, 8);
  if (vec4) k_xw_scan<64, true, true, false><<<blocks, 256, 0, st>>>(x, N, K, nullptr, nullptr, 0, xs.cnt, xs.ell_col, xs.ell_val);
  else k_xw_scan<64, false, true, false><<<blocks, 256, 0, st>>>(x, N, K, nullptr, nullptr, 0, xs.cnt, xs.ell_col, xs.ell_val);
  BIGCN_CHECK_LAUNCH("k_xw_scan (capture only)");
  return 0;
}

// y = x * wt from the CSR of x (sparse input: the dense matrix never reaches the device).
// Warp per row; the row's (col, val) pairs are fetched 32 at a time, then one fma chain per
// output in CSR order (ascending columns).
template <int NOUT>
__global__ void __launch_bounds__(256) k_xw_csr(XSparse xs, const float* __restrict__ wt, float* __restrict__ y,
                                                int64_t ldy, const int32_t* __restrict__ state) {
  constexpr int V = NOUT / 32;
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarp = ((int64_t)gridDim.x * blockDim.x) >> 5;
  // a CSR compacted from a capture that overflowed the sparse layout (BIGCN_FLAG_X_NOT_SPARSE is set) is not
  // walkable: the product is NaN, never a silent wrong answer and never an out-of-bounds read
  const bool bad = state != nullptr && state[1] != 0;
  for (int64_t row = warp0; row < xs.N; row += nwarp) {
    const int s = bad ? 0 : xs.ptr[row], e = bad ? 0 : xs.ptr[row + 1];
    float acc[V];
#pragma unroll
    for (int j = 0; j < V; ++j) acc[j] = 0.f;
    for (int p0 = s; p0 < e; p0 += 32) {
      const int p = p0 + lane;
      int k = 0;
      float v = 0.f;
      if (p < e) {
        k = xs.col[p];
        v = xs.val[p];
        if (k < 0 || k >= xs.K) {   // flagged by k_xs_from_csr / k_root_nz_csr; contributes nothing
          k = 0;
          v = 0.f;
        }
      }
      const int m = min(32, e - p0);
      for (int l = 0; l < m; ++l) {
        const int kk = __shfl_sync(FULL_MASK, k, l);
        const float vv = __shfl_sync(FULL_MASK, v, l);
        const float* wr = wt + (int64_t)kk * NOUT + lane * V;
        if (V == 4) {
          const float4 w = *reinterpret_cast<const float4*>(wr);
          fma2(acc[0], acc[1], vv, w.x, w.y);
          fma2(acc[2], acc[3], vv, w.z, w.w);
        } else {
          const float2 w = *reinterpret_cast<const float2*>(wr);
          fma2(acc[0], acc[1], vv, w.x, w.y);
        }
      }
    }
    if (bad) {
#pragma unroll
      for (int j = 0; j < V; ++j) acc[j] = __int_as_float(0x7fc00000);
    }
    float* yr = y + row * ldy + lane * V;
    if (V == 4)
      *reinterpret_cast<float4*>(yr) = make_float4(acc[0], acc[1], acc[2], acc[3]);
    else
      *reinterpret_cast<float2*>(yr) = make_float2(acc[0], acc[1]);
  }
}

// y = x * wt straight from the ELL capture of bigcn_batch_prepare (no CSR yet: the compaction runs beside this
// kernel, in the consuming step).  Rows with at most XS_ELL non-zeros walk their captured (col, val) slots -- the
// order of the fused scan, hence the same sums bit for bit; the few longer rows re-read their dense row in that
// same order (128-column strips, component-major inside a strip).
template <int NOUT>
__global__ void __launch_bounds__(256) k_xw_ell(const int32_t* __restrict__ cnt, const int32_t* __restrict__ ell_col,
                                                const float* __restrict__ ell_val, const float* __restrict__ x, int64_t N,
                                                int64_t K, const float* __restrict__ wt, float* __restrict__ y, int64_t ldy) {
  constexpr int V = NOUT / 32;
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarp = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t row = warp0; row < N; row += nwarp) {
    const int c = cnt[row];
    float acc[V];
#pragma unroll
    for (int j = 0; j < V; ++j) acc[j] = 0.f;
    auto add = [&](int64_t k, float val) {
      const float* wr = wt + k * NOUT + lane * V;
      if (V == 4) {
        const float4 w = *reinterpret_cast<const float4*>(wr);
        fma2(acc[0], acc[1], val, w.x, w.y);
        fma2(acc[2], acc[3], val, w.z, w.w);
      } else {
        const float2 w = *reinterpret_cast<const float2*>(wr);
        fma2(acc[0], acc[1], val, w.x, w.y);
      }
    };
    if (c <= XS_ELL) {
      int k = 0;
      float v = 0.f;
      if (lane < c) {
        k = ell_col[row * XS_ELL + lane];
        v = ell_val[row * XS_ELL + lane];
      }
      for (int l = 0; l < c; ++l) add(__shfl_sync(FULL_MASK, k, l), __shfl_sync(FULL_MASK, v, l));
    } else {
      const float* xr = x + row * K;
      for (int64_t s0 = 0; s0 < K; s0 += 128) {
        float comp[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int64_t kk = s0 + lane * 4 + q;
          comp[q] = kk < K ? __ldg(xr + kk) : 0.f;
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          unsigned m = __ballot_sync(FULL_MASK, comp[q] != 0.f);
          while (m) {
            const int sl = __ffs(m) - 1;
            m &= m - 1;
            add(s0 + sl * 4 + q, __shfl_sync(FULL_MASK, comp[q], sl));
          }
        }
      }
    }
    float* yr = y + row * ldy + lane * V;
    if (V == 4)
      *reinterpret_cast<float4*>(yr) = make_float4(acc[0], acc[1], acc[2], acc[3]);
    else
      *reinterpret_cast<float2*>(yr) = make_float2(acc[0], acc[1]);
  }
}
int xw_ell(const XSparse& xs, const float* x, const float* wt, int n_out, float* y, int64_t ldy, cudaStream_t st) {
  if (xs.N == 0) return 0;
  int blocks = (int)ceil_div(xs.N, 8);
  const int cap = num_sms() * 8;
  if (blocks > cap) blocks = cap;
  if (n_out == 128) k_xw_ell<128><<<blocks, 256, 0, st>>>(xs.cnt, xs.ell_col, xs.ell_val, x, xs.N, xs.K, wt, y, ldy);
  else k_xw_ell<64><<<blocks, 256, 0, st>>>(xs.cnt, xs.ell_col, xs.ell_val, x, xs.N, xs.K, wt, y, ldy);
  BIGCN_CHECK_LAUNCH("k_xw_ell");
  return 0;
}

int xw_csr(const XSparse& xs, const float* wt, int n_out, float* y, int64_t ldy, cudaStream_t st, bool check_state) {
  if (xs.N == 0) return 0;
  int blocks = (int)ceil_div(xs.N, 8);
  const int cap = num_sms() * 8;
  if (blocks > cap) blocks = cap;
  const int32_t* state = check_state ? xs.state : nullptr;
  if (n_out == 128) k_xw_csr<128><<<blocks, 256, 0, st>>>(xs, wt, y, ldy, state);
  else k_xw_csr<64><<<blocks, 256, 0, st>>>(xs, wt, y, ldy, state);
  BIGCN_CHECK_LAUNCH("k_xw_csr");
  return 0;
}

// The input gradient of k_xw_csr sampled at x's stored entries (an SDDMM): for entry e = (i, k) of the CSR,
// dval[e] = sum_o t[i][o] * wt[k][o], o < NOUT -- the dense dX = T W at the entries the forward read.
// Work units: a row's entries up to the next multiple of DXC_SEG (one unit per row), plus, for each multiple of
// DXC_SEG inside [0, ptr[N]), the entries from there to the next multiple in the row that crosses it (found by
// binary search): no unit holds more than DXC_SEG entries, so a row with all K columns spreads over many warps.
// A warp keeps its row of t in registers, takes 32 entries at a time and forms each one's dot product as lane
// partials (fixed FMA order) plus the xor butterfly of warp_sum; one store per 32 entries.  No atomics: every
// value is the same fixed-order sum on every run.  A column outside [0, K) gets 0 (the forward skips it), and so
// does every e in [ptr[N], nnz).
constexpr int DXC_SEG = 256;
constexpr int DXC_BLOCKS_PER_SM = 6;   // 40 registers, no spills (the default bound squeezes it to 32 and spills)
template <int NOUT>
__global__ void __launch_bounds__(256, DXC_BLOCKS_PER_SM)
    k_dx_csr(const int32_t* __restrict__ ptr, const int32_t* __restrict__ col, int64_t N, int64_t K, int64_t nnz,
             const float* __restrict__ t, const float* __restrict__ wt, float* __restrict__ dval) {
  // N < 2^30, nnz < 2^31 - DXC_SEG (checked by dx_csr): row, entry and unit indices fit int32
  constexpr int V = NOUT / 32;
  const int lane = threadIdx.x & 31;
  const int tid = blockIdx.x * blockDim.x + threadIdx.x, nthr = gridDim.x * blockDim.x;
  const int n = (int)N;
  const int tot = n > 0 ? (int)min((int64_t)ptr[n], nnz) : 0;   // entries that belong to a row
  for (int e = max(tot, 0) + tid; e < nnz; e += nthr) dval[e] = 0.f;
  const int nbound = tot > 0 ? (tot - 1) / DXC_SEG : 0;         // multiples of DXC_SEG strictly inside (0, tot)
  for (int u = tid >> 5; u < n + nbound; u += nthr >> 5) {
    int row, s, e;
    if (u < n) {
      row = u;
      s = ptr[row];
      e = min(ptr[row + 1], (s / DXC_SEG + 1) * DXC_SEG);
    } else {
      s = (u - n + 1) * DXC_SEG;
      int lo = 0, hi = n - 1;   // the last row starting at or before s
      while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (ptr[mid] <= s) lo = mid;
        else hi = mid - 1;
      }
      row = lo;
      if (ptr[row] == s) continue;   // the row starts on the boundary: its own unit covers these entries
      e = min(ptr[row + 1], s + DXC_SEG);
    }
    e = min(e, tot);
    if (s >= e) continue;
    float tr[V];
    {
      const float* tp = t + (int64_t)row * NOUT + lane * V;
      if (V == 4) {
        const float4 v = *reinterpret_cast<const float4*>(tp);
        tr[0] = v.x; tr[1] = v.y; tr[2] = v.z; tr[3] = v.w;
      } else {
        const float2 v = *reinterpret_cast<const float2*>(tp);
        tr[0] = v.x; tr[1] = v.y;
      }
    }
    for (int p0 = s; p0 < e; p0 += 32) {
      const int p = p0 + lane;
      const int k = p < e ? col[p] : -1;
      const int m = min(32, e - p0);
      float mine = 0.f;
      for (int l0 = 0; l0 < m; l0 += 4) {
        float part[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {   // four independent L2 reads of wt rows in flight
          const int kk = __shfl_sync(FULL_MASK, k, (l0 + j) & 31);
          part[j] = 0.f;
          if (l0 + j < m && kk >= 0 && kk < K) {   // warp-uniform
            const float* wr = wt + (int64_t)kk * NOUT + lane * V;
            if (V == 4) {
              const float4 w = *reinterpret_cast<const float4*>(wr);
              part[j] = fmaf(tr[3], w.w, fmaf(tr[2], w.z, fmaf(tr[1], w.y, tr[0] * w.x)));
            } else {
              const float2 w = *reinterpret_cast<const float2*>(wr);
              part[j] = fmaf(tr[1], w.y, tr[0] * w.x);
            }
          }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float v = warp_sum(part[j]);
          if (lane == l0 + j) mine = v;
        }
      }
      if (p < e) dval[p] = mine;
    }
  }
}
int dx_csr(const int32_t* ptr, const int32_t* col, int64_t N, int64_t K, int64_t nnz, const float* t, const float* wt,
           int n_out, float* dval, cudaStream_t st) {
  BIGCN_CHECK_ARG(N >= 0 && N < (1ll << 30) && nnz >= 0 && nnz < (1ll << 31) - DXC_SEG, "x_dgrad_csr: N or nnz too large");
  if (N == 0 && nnz == 0) return 0;
  int64_t blocks = ceil_div(N + nnz / DXC_SEG + 1, 8);
  const int64_t cap = (int64_t)num_sms() * DXC_BLOCKS_PER_SM;   // all resident: one wave of the grid-stride loop
  if (blocks > cap) blocks = cap;
  if (n_out == 128) k_dx_csr<128><<<(int)blocks, 256, 0, st>>>(ptr, col, N, K, nnz, t, wt, dval);
  else k_dx_csr<64><<<(int)blocks, 256, 0, st>>>(ptr, col, N, K, nnz, t, wt, dval);
  BIGCN_CHECK_LAUNCH("k_dx_csr");
  return 0;
}

// ------------------------------------------------------------ weight transposes
// wt[k*ldwt + col0 + o] = w[o*ldw + k0 + k], o < 64  (32 x 64 tiles through smem)
__global__ void k_transpose_w(const float* __restrict__ w, int64_t ldw, int64_t k0, int64_t K,
                              float* __restrict__ wt, int64_t ldwt, int64_t col0) {
  __shared__ float t[64][33];
  const int64_t kb = (int64_t)blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 256 threads: ty 0..7
  for (int o = ty; o < 64; o += 8) {
    const int64_t k = kb + tx;
    t[o][tx] = k < K ? w[o * ldw + k0 + k] : 0.f;
  }
  __syncthreads();
  for (int kk = ty; kk < 32; kk += 8) {
    const int64_t k = kb + kk;
    if (k < K) {
      wt[k * ldwt + col0 + tx] = t[tx][kk];
      wt[k * ldwt + col0 + 32 + tx] = t[tx + 32][kk];
    }
  }
}

// several transposes in one launch (blockIdx.y = job): the per-step weight re-layout
__global__ void k_transpose_jobs(TransposeJobs js) {
  const TransposeJob& j = js.job[blockIdx.y];
  __shared__ float t[64][33];
  const int64_t kb = (int64_t)blockIdx.x * 32;
  if (kb >= j.K) return;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int o = ty; o < 64; o += 8) {
    const int64_t k = kb + tx;
    t[o][tx] = k < j.K ? j.w[o * j.ldw + j.k0 + k] : 0.f;
  }
  __syncthreads();
  for (int kk = ty; kk < 32; kk += 8) {
    const int64_t k = kb + kk;
    if (k < j.K) {
      j.wt[k * j.ldwt + j.col0 + tx] = t[tx][kk];
      j.wt[k * j.ldwt + j.col0 + 32 + tx] = t[tx + 32][kk];
    }
  }
}
int transpose_jobs_launch(const TransposeJobs& js, cudaStream_t st) {
  int64_t kmax = 0;
  for (int i = 0; i < js.n; ++i) kmax = js.job[i].K > kmax ? js.job[i].K : kmax;
  if (js.n == 0 || kmax == 0) return 0;
  k_transpose_jobs<<<dim3((int)ceil_div(kmax, 32), js.n), 256, 0, st>>>(js);
  BIGCN_CHECK_LAUNCH("k_transpose_jobs");
  return 0;
}

int transpose_weight(const float* w, int64_t ldw, int64_t k0, int64_t K, float* wt, int64_t ldwt,
                     int64_t col0, cudaStream_t st) {
  if (K == 0) return 0;
  k_transpose_w<<<(int)ceil_div(K, 32), 256, 0, st>>>(w, ldw, k0, K, wt, ldwt, col0);
  BIGCN_CHECK_LAUNCH("k_transpose_w");
  return 0;
}

// ------------------------------------------------------- gT[k, :] = sum_i x[i,k] * t[i, :]
// CTA = one 16-column slab of X (64 B = 2 sectors per row) x one chunk of rows.  EVERY warp
// covers all 16 columns for its own rows and keeps the 16 x NOUT accumulators in registers,
// so a column that is non-zero in every row (common words in a bag-of-words matrix) costs the
// same as any other: its hits are spread over all warps of all row chunks instead of
// serialising in one owner.  X never passes through registers: each warp streams 64-row
// stages (4 KB) into its private shared-memory ring with cp.async (two stages, 16 B per
// lane), ballots the non-zero rows of a landed stage, fetches the T rows of up to four hit
// rows at once (L2) and adds x[row][c] * T[row][:] for the non-zero c, broadcast-reading the
// row's 16 values from shared memory.  Per column the contributions arrive in ascending row
// order inside a warp, warps are combined in index order, row chunks in order by
// k_dw_reduce: no atomics, bit-reproducible.
constexpr int DW_U = 8;                         // cp.async per lane per stage
constexpr int DW_COLS = 16;
constexpr int DW_WARP_ROWS = 8 * DW_U;          // 64 rows per stage
constexpr int DW_CTA_ROWS = 8 * DW_WARP_ROWS;   // 512 rows per CTA pass
constexpr int DW_STAGE_FLOATS = DW_WARP_ROWS * DW_COLS;  // 1024
constexpr int DW_SMEM_BYTES = 8 * 2 * DW_STAGE_FLOATS * 4;  // 64 KB

__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gsrc, int src_bytes) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(d), "l"(gsrc), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N_>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N_)); }

template <int NOUT>
__global__ void __launch_bounds__(256, 2) k_dw_slab(const float* __restrict__ x, int64_t N, int64_t K,
                                                    const float* __restrict__ t, int64_t ldt,
                                                    float* __restrict__ partial, int rows_per_chunk) {
  constexpr int V = NOUT / 32;
  extern __shared__ __align__(16) float dw_smem[];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  float* xs = dw_smem + (size_t)w * 2 * DW_STAGE_FLOATS;
  const int64_t c0 = (int64_t)blockIdx.x * DW_COLS;
  const int64_t r_begin = (int64_t)blockIdx.y * rows_per_chunk;
  const int64_t r_end = min(N, r_begin + rows_per_chunk);
  const int q = lane & 3;    // which float4 of the slab
  const int rl = lane >> 2;  // row within the 8-row group
  const int64_t col = c0 + q * 4;
  const bool col_ok = col < K;  // K % 4 == 0 -> whole float4 valid
  float acc[DW_COLS][V];
#pragma unroll
  for (int c = 0; c < DW_COLS; ++c)
#pragma unroll
    for (int j = 0; j < V; ++j) acc[c][j] = 0.f;

  auto issue = [&](int stage, int64_t rb) {
#pragma unroll
    for (int u = 0; u < DW_U; ++u) {
      const int64_t r = rb + u * 8 + rl;
      const bool ok = col_ok && r < r_end;
      cp_async16(xs + stage * DW_STAGE_FLOATS + (u * 32 + lane) * 4, ok ? x + r * K + col : x, ok ? 16 : 0);
    }
    cp_async_commit();
  };

  int64_t rb = r_begin + (int64_t)w * DW_WARP_ROWS;
  int stage = 0;
  if (rb < r_end) issue(0, rb);
  for (; rb < r_end; rb += DW_CTA_ROWS, stage ^= 1) {
    const bool more = rb + DW_CTA_ROWS < r_end;
    if (more) {
      issue(stage ^ 1, rb + DW_CTA_ROWS);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncwarp();
    const float* st = xs + stage * DW_STAGE_FLOATS;
    // which of the 64 rows of this stage hold a non-zero
    unsigned long long hits = 0ull;
#pragma unroll
    for (int u = 0; u < DW_U; ++u) {
      const float4 v = *reinterpret_cast<const float4*>(st + (u * 32 + lane) * 4);
      const bool any = (v.x != 0.f) | (v.y != 0.f) | (v.z != 0.f) | (v.w != 0.f);
      unsigned m = __ballot_sync(FULL_MASK, any);
      m |= m >> 1;
      m |= m >> 2;
      m &= 0x11111111u;   // bit 4*rr set <=> row rr hit
      m = (m | (m >> 3)) & 0x03030303u;
      m = (m | (m >> 6)) & 0x000f000fu;
      m = (m | (m >> 12)) & 0xffu;
      hits |= (unsigned long long)m << (u * 8);
    }
    const float* trow = t + rb * ldt + lane * V;
    while (hits) {
      int rows[4];
      float tv[4][V];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        rows[j] = -1;
        if (hits) {
          rows[j] = __ffsll((long long)hits) - 1;
          hits &= hits - 1;
          if (V == 4) {
            const float4 g = *reinterpret_cast<const float4*>(trow + (int64_t)rows[j] * ldt);
            tv[j][0] = g.x; tv[j][1] = g.y; tv[j][2] = g.z; tv[j][3] = g.w;
          } else {
            const float2 g = *reinterpret_cast<const float2*>(trow + (int64_t)rows[j] * ldt);
            tv[j][0] = g.x; tv[j][1] = g.y;
          }
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (rows[j] < 0) continue;
        const float4* xr = reinterpret_cast<const float4*>(st + rows[j] * DW_COLS);
#pragma unroll
        for (int qq = 0; qq < 4; ++qq) {
          const float4 xv = xr[qq];   // broadcast read
          const float xa[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
          for (int c = 0; c < 4; ++c)
            if (xa[c] != 0.f) {
#pragma unroll
              for (int jj = 0; jj < V; ++jj) acc[qq * 4 + c][jj] = fmaf(xa[c], tv[j][jj], acc[qq * 4 + c][jj]);
            }
        }
      }
    }
    __syncwarp();
  }
  // ordered combine of the 8 warps (reusing the ring), then one coalesced store of the slab's partial
  __syncthreads();
  float* red = dw_smem;
  for (int ww = 0; ww < 8; ++ww) {
    if (w == ww) {
#pragma unroll
      for (int c = 0; c < DW_COLS; ++c)
#pragma unroll
        for (int j = 0; j < V; ++j) {
          float* p = red + c * NOUT + lane * V + j;
          *p = (ww == 0) ? acc[c][j] : (*p + acc[c][j]);
        }
    }
    __syncthreads();
  }
  float* out = partial + ((size_t)blockIdx.y * K) * NOUT;
  for (int i = threadIdx.x; i < DW_COLS * NOUT; i += 256) {
    const int64_t k = c0 + i / NOUT;
    if (k < K) out[k * NOUT + (i % NOUT)] = red[i];
  }
}

// scalar fallback for K % 4 != 0 or unaligned x: thread per (k, o) pair, rows in order
template <int NOUT>
__global__ void k_dw_naive(const float* __restrict__ x, int64_t N, int64_t K,
                           const float* __restrict__ t, int64_t ldt, float* __restrict__ partial) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= K * NOUT) return;
  const int64_t k = idx / NOUT;
  const int o = (int)(idx % NOUT);
  float acc = 0.f;
  for (int64_t i = 0; i < N; ++i) {
    const float xv = x[i * K + k];
    if (xv != 0.f) acc = fmaf(xv, t[i * ldt + o], acc);
  }
  partial[k * NOUT + o] = acc;
}

// dw[o*ldw + k0 + k] = sum_chunk partial[chunk][k][col0 + o]   (o < 64), chunks in order
__global__ void k_dw_reduce(const float* __restrict__ partial, int nchunk, int64_t K, int nout,
                            float* __restrict__ dw_a, int64_t ldw_a, int64_t k0_a,
                            float* __restrict__ dw_b, int64_t ldw_b, int64_t k0_b) {
  __shared__ float tile[32][65];
  // blockIdx.y = which 64-output half (direction) of the partials
  const int col0 = blockIdx.y * 64;
  float* __restrict__ dw = blockIdx.y ? dw_b : dw_a;
  const int64_t ldw = blockIdx.y ? ldw_b : ldw_a;
  const int64_t k0 = blockIdx.y ? k0_b : k0_a;
  const int64_t kb = (int64_t)blockIdx.x * 32;
  const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;  // 256 threads: 4 x 64
  for (int kk = ty; kk < 32; kk += 4) {
    const int64_t k = kb + kk;
    float s = 0.f;
    if (k < K)
      for (int c = 0; c < nchunk; ++c) s += partial[((size_t)c * K + k) * nout + col0 + tx];
    tile[kk][tx] = s;
  }
  __syncthreads();
  const int lx = threadIdx.x & 31, ly = threadIdx.x >> 5;  // 8 x 32
  for (int o = ly; o < 64; o += 8) {
    const int64_t k = kb + lx;
    if (k < K) dw[o * ldw + k0 + k] = tile[lx][o];
  }
}

struct DwPlan {
  int nchunk;
  int rows_per_chunk;
  bool fast;
};
DwPlan dw_plan(int64_t N, int64_t K, const float* x) {
  DwPlan p;
  p.fast = (K % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  if (!p.fast) {
    p.nchunk = 1;
    p.rows_per_chunk = (int)N;
    return p;
  }
  const int64_t slabs = ceil_div(K, DW_COLS);
  int64_t want = ceil_div((int64_t)num_sms() * 8, slabs);
  const int64_t max_chunks = ceil_div(N, DW_CTA_ROWS);  // at least one full CTA pass per chunk
  if (want > max_chunks) want = max_chunks;
  if (want < 1) want = 1;
  int64_t rpc = ceil_div(N, want);
  rpc = ceil_div(rpc, DW_WARP_ROWS) * DW_WARP_ROWS;
  p.rows_per_chunk = (int)rpc;
  p.nchunk = (int)ceil_div(N, rpc);
  return p;
}
size_t dw_partial_floats(int64_t N, int64_t K, int n_out) {
  // upper bound independent of the pointer alignment
  const int64_t slabs = ceil_div(K, DW_COLS);
  int64_t want = ceil_div((int64_t)num_sms() * 8, slabs > 0 ? slabs : 1);
  if (want < 1) want = 1;
  const size_t scan = (size_t)(want + 1) * (size_t)K * (size_t)n_out;
  const size_t tc = (size_t)(num_sms() + 1) * 256 * (size_t)n_out;   // tcgen05 split-K partials (gemm_tc.cu)
  return scan > tc ? scan : tc;
}

// grad of x*wt wrt the weights: writes dw_a (cols [0,64) of t) and, if n_out == 128, dw_b (cols [64,128))
int dw_fp32(const float* x, int64_t N, int64_t K, const float* t, int64_t ldt, int n_out,
            float* partial, float* dw_a, int64_t ldw_a, int64_t k0_a, float* dw_b, int64_t ldw_b,
            int64_t k0_b, cudaStream_t st) {
  if (K == 0) return 0;
  if (N == 0) {   // before dw_plan, whose chunk size is 0 rows here
    cudaMemsetAsync(partial, 0, (size_t)K * n_out * sizeof(float), st);
    return dw_reduce_launch(partial, 1, K, n_out, dw_a, ldw_a, k0_a, dw_b, ldw_b, k0_b, st);
  }
  const DwPlan p = dw_plan(N, K, x);
  if (p.fast) {
    dim3 grid((unsigned)ceil_div(K, DW_COLS), (unsigned)p.nchunk);
    static bool attr_set = false;
    if (!attr_set) {
      cudaFuncSetAttribute(k_dw_slab<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, DW_SMEM_BYTES);
      cudaFuncSetAttribute(k_dw_slab<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, DW_SMEM_BYTES);
      attr_set = true;
    }
    if (n_out == 128) {
      k_dw_slab<128><<<grid, 256, DW_SMEM_BYTES, st>>>(x, N, K, t, ldt, partial, p.rows_per_chunk);
    } else {
      k_dw_slab<64><<<grid, 256, DW_SMEM_BYTES, st>>>(x, N, K, t, ldt, partial, p.rows_per_chunk);
    }
    BIGCN_CHECK_LAUNCH("k_dw_slab");
  } else {
    const int64_t tot = K * n_out;
    if (n_out == 128) k_dw_naive<128><<<(int)ceil_div(tot, 256), 256, 0, st>>>(x, N, K, t, ldt, partial);
    else k_dw_naive<64><<<(int)ceil_div(tot, 256), 256, 0, st>>>(x, N, K, t, ldt, partial);
    BIGCN_CHECK_LAUNCH("k_dw_naive");
  }
  return dw_reduce_launch(partial, p.nchunk, K, n_out, dw_a, ldw_a, k0_a, dw_b, ldw_b, k0_b, st);
}

int dw_reduce_launch(const float* partial, int nchunk, int64_t K, int n_out, float* dw_a, int64_t ldw_a,
                     int64_t k0_a, float* dw_b, int64_t ldw_b, int64_t k0_b, cudaStream_t st) {
  const int halves = (n_out == 128 && dw_b != nullptr) ? 2 : 1;
  k_dw_reduce<<<dim3((int)ceil_div(K, 32), halves), 256, 0, st>>>(partial, nchunk, K, n_out, dw_a, ldw_a, k0_a,
                                                                  dw_b, ldw_b, k0_b);
  BIGCN_CHECK_LAUNCH("k_dw_reduce");
  return 0;
}

}  // namespace bigcn

extern "C" int bigcn_transpose_weight(const float* w, int64_t ldw, int64_t k0, int64_t K, float* wt,
                                      int64_t ldwt, int64_t col0, bigcn_stream_t stream) {
  return bigcn::transpose_weight(w, ldw, k0, K, wt, ldwt, col0, reinterpret_cast<cudaStream_t>(stream));
}
