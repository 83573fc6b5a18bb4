// tcgen05 / TMA / TMEM building blocks shared by the tensor-core kernels (gemm_tc.cu: X * W^T and dW1;
// mix_tc.cu: the 64 x 64 contractions of conv2.lin and its backward).  sm_100a only.
#pragma once
#include <cuda.h>

#include "kernels.cuh"

namespace bigcn {

// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor):
//   [0,14) start address >> 4, [16,30) LBO >> 4 (= 1, unused for swizzled K-major),
//   [32,46) SBO >> 4 (1024 B between 8-row groups), [46,48) version = 1, [61,64) layout = 2 (SW128)
__device__ __forceinline__ uint64_t make_desc_k_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// kind::tf32 instruction descriptor (cute::UMMA::InstrDescriptor): c_format F32 (1) at [4,6),
// a/b_format TF32 (2) at [7,10)/[10,13), K-major A and B, N >> 3 at [17,23), M >> 4 at [24,29)
__host__ __device__ constexpr uint32_t make_idesc_tf32(int m, int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// ---- kind::f16 (BIGCN_GEMM_BF16: bf16 operands, fp32 accumulator in TMEM), UMMA_K = 16
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// kind::f16 instruction descriptor: c_format F32 (1) at [4,6), a/b_format BF16 (1) at [7,10)/[10,13), K-major A and B,
// N >> 3 at [17,23), M >> 4 at [24,29)
__host__ __device__ constexpr uint32_t make_idesc_bf16(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
// K-major SWIZZLE_64B descriptor: rows of 64 B (32 bf16), 8-row atoms of 512 B (SBO), LBO unused, layout 4 (SW64)
__device__ __forceinline__ uint64_t make_desc_k_sw64(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(512 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)4 << 61;
  return d;
}
// MN-major SWIZZLE_128B descriptor for 16-bit operands: 128 B (64 bf16) contiguous along MN, rows of the K axis 128 B
// apart, 8-row atoms (SBO = 1024 B), LBO = bytes between 64-element MN blocks
__device__ __forceinline__ uint64_t make_desc_mn_sw128_16b(uint32_t saddr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;   // LayoutType::SWIZZLE_128B
  return d;
}

// generic-proxy writes to shared memory -> visible to the async proxy (tcgen05.mma reads)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Converter warps (cw = 0..3 of 4): split `bytes` of fp32 at `x_smem` into hi (in place, low 13 mantissa bits
// cleared: exactly what a TF32 MMA can represent) and lo = tf32(x - hi) at `lo_smem`.  Position-preserving, so
// the TMA swizzle of the tile carries over (both buffers are 1024 B aligned).
// lo = (x - hi) rounded to the nearest TF32 (a truncated lo leaves a residual with the sign of x: a bias that column
// sums over thousands of rows would accumulate)
__device__ __forceinline__ uint32_t tf32_lo_bits(uint32_t x, uint32_t hi) {
  return (__float_as_uint(__uint_as_float(x) - __uint_as_float(hi)) + 0x1000u) & 0xFFFFE000u;
}
__device__ __forceinline__ void split_tile_hi_lo(uint32_t x_smem, uint32_t lo_smem, int bytes, int cw, int lane) {
  for (int off = (cw * 32 + lane) * 16; off < bytes; off += 128 * 16) {
    uint32_t a, b, c, d;
    asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(x_smem + off));
    const uint32_t ha = a & 0xFFFFE000u, hb = b & 0xFFFFE000u, hc = c & 0xFFFFE000u, hd = d & 0xFFFFE000u;
    const uint32_t la = tf32_lo_bits(a, ha), lb = tf32_lo_bits(b, hb), lc = tf32_lo_bits(c, hc), ld = tf32_lo_bits(d, hd);
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(x_smem + off), "r"(ha), "r"(hb), "r"(hc), "r"(hd) : "memory");
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(lo_smem + off), "r"(la), "r"(lb), "r"(lc), "r"(ld) : "memory");
  }
}


// ---------------------------------------------------------------- host side: tensor maps
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// 2-D fp32 row-major [rows, cols] with row pitch ld (elements); box = 32 cols x box_rows, SW128
inline int make_map(CUtensorMap* m, const float* base, int64_t rows, int64_t cols, int64_t ld, int box_rows) {
  const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t gstr[1] = {(cuuint64_t)ld * 4};
  const cuuint32_t box[2] = {32, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = encode_fn()(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim, gstr, box,
                                 estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                 CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("xw_tc: cuTensorMapEncodeTiled failed (%d)", (int)r);
    return 2;
  }
  return 0;
}

// 2-D bf16 row-major [rows, cols] with row pitch ld (elements); box = box_cols x box_rows with the given swizzle
inline int make_map_bf16(CUtensorMap* m, const void* base, int64_t rows, int64_t cols, int64_t ld, int box_cols,
                         int box_rows, CUtensorMapSwizzle swizzle) {
  const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t gstr[1] = {(cuuint64_t)ld * 2};
  const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = encode_fn()(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr, box,
                                 estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                 CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("bf16 tensor map: cuTensorMapEncodeTiled failed (%d)", (int)r);
    return 2;
  }
  return 0;
}


}  // namespace bigcn
