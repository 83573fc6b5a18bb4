// Shared device helpers for libbigcn_b200.so (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/bigcn_b200.h"

#define H BIGCN_H
#define FULL_MASK 0xffffffffu

namespace bigcn {

void set_error(const char* fmt, ...);
int num_sms();

#define BIGCN_CHECK_ARG(cond, ...)          \
  do {                                      \
    if (!(cond)) {                          \
      bigcn::set_error(__VA_ARGS__);        \
      return 1;                             \
    }                                       \
  } while (0)

#define BIGCN_CHECK_LAUNCH(name)                                                        \
  do {                                                                                  \
    cudaError_t e__ = cudaGetLastError();                                               \
    if (e__ != cudaSuccess) {                                                           \
      bigcn::set_error("%s: launch failed: %s", name, cudaGetErrorString(e__));         \
      return 2;                                                                         \
    }                                                                                   \
  } while (0)

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Bump allocator over a caller-provided workspace (256 B aligned slices).
struct Carver {
  char* base;
  size_t off = 0;
  size_t cap;
  Carver(void* p, size_t bytes) : base(reinterpret_cast<char*>(p)), cap(bytes) {}
  template <typename T>
  T* take(size_t n) {
    off = align_up(off, 256);
    T* r = reinterpret_cast<T*>(base ? base + off : nullptr);
    off += n * sizeof(T);
    return r;
  }
  bool ok() const { return off <= cap; }
};

// ---------------------------------------------------------------- device side
__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

// an element of x as fp32: x is fp32, or bf16 in BIGCN_GEMM_BF16 (widened exactly)
__device__ __forceinline__ float x_f32(float v) { return v; }
__device__ __forceinline__ float x_f32(__nv_bfloat16 v) { return __bfloat162float(v); }

__device__ __forceinline__ float4 ldg_stream_f4(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}

// the same with an L2 evict-first policy: x is read once per step and must not push the L2-resident activation
// panels ([N,64] H1 / A1 / Z / T ...) of the step's other kernels out of the 126 MB L2
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ float4 ldg_stream_f4_ef(const float* p, uint64_t pol) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p), "l"(pol));
  return r;
}

// Two independent IEEE fp32 fmas in ONE instruction (sm_100 FFMA2, scalar x pair + pair): (z0, z1) = s * (w0, w1) + (z0, z1).
// Same results bit for bit as two fmaf(); half the issue slots -- the sweeps and 64 x 64 products here are issue-bound.
// (mul.rn.f32x2 + add.rn.f32x2 is NOT used for the separately-rounded sums of the EXACT sweeps: ptxas contracts the pair.)
__device__ __forceinline__ void fma2(float& z0, float& z1, float s, float w0, float w1) {
  unsigned long long a, b, c, d;
  asm("mov.b64 %0, {%1, %1};" : "=l"(a) : "f"(s));
  asm("mov.b64 %0, {%1, %2};" : "=l"(b) : "f"(w0), "f"(w1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(c) : "f"(z0), "f"(z1));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(z0), "=f"(z1) : "l"(d));
}
__device__ __forceinline__ void fma4(float4& z, float s, const float4& w) {
  fma2(z.x, z.y, s, w.x, w.y);
  fma2(z.z, z.w, s, w.z, w.w);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL_MASK, v, o);
  return v;
}

// ---- mbarrier / bulk-copy (TMA engine, UBLKCP) primitives ----------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  }
}
// global -> shared bulk copy (bytes % 16 == 0, both addresses 16 B aligned), completion counted
// in bytes on the mbarrier
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}

// the same with an L2 cache policy (evict-first for data that is read exactly once)
__device__ __forceinline__ void bulk_g2s_hint(uint32_t dst_smem, const void* src, uint32_t bytes, uint32_t bar, uint64_t pol) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst_smem),
               "l"(src), "r"(bytes), "r"(bar), "l"(pol)
               : "memory");
}

// Philox4x32-10 (Salmon et al. SC'11); spec mirrored by oracle/gcn_oracle.py.
struct Philox4 {
  uint32_t x, y, z, w;
};
__device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                  uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return Philox4{c0, c1, c2, c3};
}

// Dropout spec: keep[node, col] = philox(ctr=(col>>2, node_lo, node_hi, stream), key=seed)[col&3] >= thresh
struct DropSpec {
  uint32_t k0, k1;     // seed
  uint32_t thresh;     // round(p * 2^32)
  uint32_t stream;     // 0 TD, 1 BU
  float scale;         // 1/(1-p)
  int32_t on;          // training
  const unsigned long long* ctr;   // device counter added to the seed (CUDA-graph replays draw fresh masks), or NULL
};
__device__ __forceinline__ Philox4 drop_block(const DropSpec& d, int64_t node, uint32_t col_block) {
  uint32_t k0 = d.k0, k1 = d.k1;
  if (d.ctr != nullptr) {   // seed + *ctr as one 64-bit sum; the counter only moves between launches
    const unsigned long long s = (((unsigned long long)k1 << 32) | k0) + __ldg(d.ctr);
    k0 = (uint32_t)s;
    k1 = (uint32_t)(s >> 32);
  }
  return philox4x32_10(col_block, (uint32_t)(node & 0xffffffffll), (uint32_t)((uint64_t)node >> 32),
                       d.stream, k0, k1);
}
__device__ __forceinline__ uint32_t philox_elem(const Philox4& r, int e) {
  return e == 0 ? r.x : (e == 1 ? r.y : (e == 2 ? r.z : r.w));
}

static inline uint32_t drop_threshold(float p) {
  double t = (double)p * 4294967296.0;
  double r = t + 0.5;
  // round-half-even to mirror Python round()
  double f = (double)(uint64_t)r;
  if (r == f && ((uint64_t)f & 1ull) && (t - (double)(uint64_t)t) == 0.5) f -= 1.0;
  if (f < 0) f = 0;
  if (f > 4294967295.0) f = 4294967295.0;
  return (uint32_t)f;
}
static inline DropSpec make_drop(const bigcn_opts_t* o, int stream_id) {
  DropSpec d;
  d.k0 = (uint32_t)(o->seed & 0xffffffffull);
  d.k1 = (uint32_t)(o->seed >> 32);
  d.thresh = drop_threshold(o->p_drop);
  d.stream = (uint32_t)stream_id;
  d.scale = 1.0f / (1.0f - o->p_drop);
  d.on = o->training && o->p_drop > 0.f;
  d.ctr = reinterpret_cast<const unsigned long long*>(o->seed_dev);
  return d;
}

}  // namespace bigcn
