// Device half of the host feeder (bigcn_b200/feeder.py): rows of a dense fp32 feature matrix that
// crossed PCIe as they are (the reference's loader hands over dense bag-of-words rows,
// Process/dataset.py:64-99) are compacted to CSR on the device, while the host compacts the other
// rows itself (host_compact.cpp); both parts land in ONE CSR the sparse input path consumes.
// Pure data movement (integer / byte work, HBM-bound): warp per row, 512 B per warp-instruction.
#include "kernels.cuh"

namespace bigcn {

__device__ __forceinline__ int nz4(const float4& v) {
  return (v.x != 0.f) + (v.y != 0.f) + (v.z != 0.f) + (v.w != 0.f);
}

// non-zeros per row
__global__ void __launch_bounds__(256) k_feed_count(const float* __restrict__ x, int64_t N, int64_t K,
                                                    int32_t* __restrict__ cnt) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarp = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const bool vec = (K % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  for (int64_t r = warp0; r < N; r += nwarp) {
    const float* xr = x + r * K;
    int c = 0;
    if (vec) {
      const int64_t k4 = K / 4;
      int64_t q = lane;
      for (; q + 96 < k4; q += 128) {          // four 512 B loads in flight
        const float4 a = ldg_stream_f4(xr + 4 * q), b = ldg_stream_f4(xr + 4 * (q + 32));
        const float4 d = ldg_stream_f4(xr + 4 * (q + 64)), e = ldg_stream_f4(xr + 4 * (q + 96));
        c += nz4(a) + nz4(b) + nz4(d) + nz4(e);
      }
      for (; q < k4; q += 32) c += nz4(ldg_stream_f4(xr + 4 * q));
    } else {
      for (int64_t k = lane; k < K; k += 32) c += xr[k] != 0.f;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(FULL_MASK, c, o);
    if (lane == 0) cnt[r] = c;
  }
}

// the same count for a bf16 x (BIGCN_GEMM_BF16's density probe): 8 elements per 16 B load when rows allow it; a bf16
// is zero when its bits other than the sign are (so -0 counts as zero, as -0.f != 0.f is false above)
__device__ __forceinline__ int nz_bf16x2(uint32_t v) { return ((v & 0x7FFFu) != 0u) + ((v & 0x7FFF0000u) != 0u); }
__global__ void __launch_bounds__(256) k_feed_count_bf16(const __nv_bfloat16* __restrict__ x, int64_t N, int64_t K,
                                                         int32_t* __restrict__ cnt) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarp = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const bool vec = (K % 8 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  for (int64_t r = warp0; r < N; r += nwarp) {
    const __nv_bfloat16* xr = x + r * K;
    int c = 0;
    if (vec) {
      for (int64_t q = lane; q < K / 8; q += 32) {
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(xr) + q);
        c += nz_bf16x2(v.x) + nz_bf16x2(v.y) + nz_bf16x2(v.z) + nz_bf16x2(v.w);
      }
    } else {
      for (int64_t k = lane; k < K; k += 32) c += __bfloat162float(xr[k]) != 0.f;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(FULL_MASK, c, o);
    if (lane == 0) cnt[r] = c;
  }
}

// second pass: (col, val) of every row in ascending column order at ptr_local[r] + base; also the
// rows' entries of the combined row-pointer array
__global__ void __launch_bounds__(256) k_feed_fill(const float* __restrict__ x, int64_t N, int64_t K,
                                                   const int32_t* __restrict__ incl /* inclusive scan of cnt */,
                                                   int32_t base, int32_t* __restrict__ ptr_out /* [N] -> ptr[row + 1] */,
                                                   int32_t* __restrict__ col, float* __restrict__ val, int64_t cap,
                                                   int32_t* __restrict__ flags) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarp = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const bool vec = (K % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  for (int64_t r = warp0; r < N; r += nwarp) {
    const float* xr = x + r * K;
    const int64_t end64 = (int64_t)incl[r] + base;
    int32_t pos = (r > 0 ? incl[r - 1] : 0) + base;
    if (end64 > cap) {                         // does not fit the arrays: the row is dropped and the caller told
      if (lane == 0) {
        ptr_out[r] = (int32_t)(pos < cap ? pos : cap);
        atomicOr(flags, BIGCN_FLAG_X_NOT_SPARSE);
      }
      continue;
    }
    const int32_t end = (int32_t)end64;
    if (lane == 0) ptr_out[r] = end;
    if (pos == end) continue;                  // empty row: nothing to write, no second read
    if (vec) {
      const int64_t k4 = K / 4;
      for (int64_t q0 = 0; q0 < k4; q0 += 32) {
        const int64_t q = q0 + lane;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (q < k4) v = ldg_stream_f4(xr + 4 * q);
        const int c = nz4(v);
        if (__ballot_sync(FULL_MASK, c != 0) == 0) continue;
        int inc = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int t = __shfl_up_sync(FULL_MASK, inc, o);
          if (lane >= o) inc += t;
        }
        int p = pos + inc - c;
        const float e[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (e[j] != 0.f) {
            col[p] = (int32_t)(4 * q + j);
            val[p] = e[j];
            ++p;
          }
        pos += __shfl_sync(FULL_MASK, inc, 31);
      }
    } else {
      for (int64_t k0 = 0; k0 < K; k0 += 32) {
        const int64_t k = k0 + lane;
        const float v = k < K ? xr[k] : 0.f;
        const unsigned m = __ballot_sync(FULL_MASK, v != 0.f);
        if (v != 0.f) {
          const int p = pos + __popc(m & ((1u << lane) - 1u));
          col[p] = (int32_t)k;
          val[p] = v;
        }
        pos += __popc(m);
      }
    }
  }
}

}  // namespace bigcn

using namespace bigcn;

static int feed_grid(int64_t N) {
  int64_t b = ceil_div(N > 0 ? N : 1, 8);
  const int64_t cap = (int64_t)num_sms() * 8;
  return (int)(b > cap ? cap : b);
}

extern "C" int bigcn_dense_row_counts(const float* x, int64_t N, int64_t K, int32_t* cnt, bigcn_stream_t stream) {
  BIGCN_CHECK_ARG(N >= 0 && K > 0 && (N == 0 || (x && cnt)), "dense_row_counts: bad arguments");
  if (N == 0) return 0;
  k_feed_count<<<feed_grid(N), 256, 0, (cudaStream_t)stream>>>(x, N, K, cnt);
  BIGCN_CHECK_LAUNCH("k_feed_count");
  return 0;
}

extern "C" int bigcn_dense_row_counts_bf16(const void* x, int64_t N, int64_t K, int32_t* cnt, bigcn_stream_t stream) {
  BIGCN_CHECK_ARG(N >= 0 && K > 0 && (N == 0 || (x && cnt)), "dense_row_counts_bf16: bad arguments");
  if (N == 0) return 0;
  k_feed_count_bf16<<<feed_grid(N), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const __nv_bfloat16*>(x), N, K, cnt);
  BIGCN_CHECK_LAUNCH("k_feed_count_bf16");
  return 0;
}

extern "C" int bigcn_dense_rows_to_csr(const float* x, int64_t N, int64_t K, const int32_t* incl_counts, int64_t base,
                                       int32_t* ptr_out, int32_t* col, float* val, int64_t cap, int32_t* flags,
                                       bigcn_stream_t stream) {
  BIGCN_CHECK_ARG(N >= 0 && K > 0 && base >= 0 && base <= cap && cap < (1ll << 31) && flags &&
                      (N == 0 || (x && incl_counts && ptr_out && col && val)), "dense_rows_to_csr: bad arguments");
  if (N == 0) return 0;
  k_feed_fill<<<feed_grid(N), 256, 0, (cudaStream_t)stream>>>(x, N, K, incl_counts, (int32_t)base, ptr_out, col, val, cap, flags);
  BIGCN_CHECK_LAUNCH("k_feed_fill");
  return 0;
}
