// CSR row sweep shared by every A-hat / A-hat^T kernel (k_propagate, k_propagate_g2, k_prop1_mix).
//
//   out[i] = post( sum_{e in ptr[i]..ptr[i+1]} (dis[idx[e]] * dis[i]) * val(idx[e])  +  dis[i]^2 * val(i) )
//   (or, edge-weighted, the precomputed normalised weight of each entry and of the self-loop: WtEntry)
//
// replaces MessagePassing.propagate of torch_geometric's GCNConv (index_select, broadcast
// multiply, atomic scatter_add) reached from BiGCN_Twitter.py:42,56,92,105 and its autograd
// transpose.  Design (measured on B200, tools/kbench.py):
//  * half-warp per block of R CONSECUTIVE rows (16 lanes x float4 = one 256 B row per
//    instruction); the block's in-edges are one contiguous CSR range, so 16 (index, weight)
//    pairs are fetched with one coalesced load each;
//  * neighbour rows and the block's own rows land in a shared-memory stage through cp.async
//    (LDGSTS): (R + Q) x 256 B in flight per half-warp without a register landing zone;
//  * warps pull units (two adjacent blocks) from a CTA-local counter, CTAs own interleaved
//    chunks of units: a heavy block delays one warp, not a whole static stripe; loop bounds are
//    warp-uniform so the two halves stay converged (one instruction stream for 2 blocks);
//  * per row the additions run in COO' order (in-edges in list order, then the self-loop) with
//    separate multiply and add when EXACT: bit-identical to the CPU index_add_ of the oracle;
//  * hub rows (more than LONG_ROW in-edges: the root of a reply tree in the child-sum direction)
//    are left out of the main sweep and split into <= LONG_MAX_CHUNKS fixed chunks that other
//    half-warps sum independently; the last arriver (device counter) adds the partials in chunk
//    order and finishes the row.  Deterministic, no floating-point atomics; only the summation
//    order of those rows differs from the sequential oracle.
#pragma once
#include "kernels.cuh"

namespace bigcn {

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, const float4& v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ float comp4(const float4& v, int c) {
  return c == 0 ? v.x : (c == 1 ? v.y : (c == 2 ? v.z : v.w));
}
__device__ __forceinline__ void wadd4(float4& acc, float w, const float4& h) {
  acc.x = __fadd_rn(acc.x, __fmul_rn(w, h.x));
  acc.y = __fadd_rn(acc.y, __fmul_rn(w, h.y));
  acc.z = __fadd_rn(acc.z, __fmul_rn(w, h.z));
  acc.w = __fadd_rn(acc.w, __fmul_rn(w, h.w));
}
template <bool EXACT>
__device__ __forceinline__ void acc_add(float4& acc, float w, const float4& v) {
  if (EXACT) {
    wadd4(acc, w, v);
  } else {
    fma4(acc, w, v);
  }
}
__device__ __forceinline__ unsigned half_mask(int half) { return half ? 0xffff0000u : 0x0000ffffu; }

__device__ __forceinline__ void cp_async_row16(float* smem_dst, const float* gsrc) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit_wait_all() {
  asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory");
}

// ---- hub-row work lists (built by graph prep, one per CSR) ---------------------------------
// Layout of the int32 blob `lng` (size long_ws_ints(E)):
//   [0] n_long  [1] n_items  [2..3] pad | done[cap_rows] | row[cap_rows] | item0[cap_rows] |
//   item_slot[cap_items] | partial[cap_items][64] (fp32, 16 B aligned)
struct LongView {
  int32_t* cnt;
  int32_t* done;
  int32_t* row;
  int32_t* item0;
  int32_t* item_slot;
  float* partial;
};
__host__ __device__ inline int64_t long_cap_rows(int64_t E) { return E / (LONG_ROW + 1) + 1; }
__host__ __device__ inline int64_t long_cap_items(int64_t E) { return E / LONG_ROW + long_cap_rows(E) + 1; }
__host__ __device__ inline int64_t long_hdr_ints(int64_t E) { return 4 + (long_cap_rows(E) + 3) / 4 * 4; }
__host__ __device__ inline int64_t long_ws_ints_impl(int64_t E) {
  const int64_t r = (long_cap_rows(E) + 3) / 4 * 4, it = (long_cap_items(E) + 3) / 4 * 4;
  return 4 + 3 * r + it + it * H;
}
__host__ __device__ inline LongView long_view(int32_t* ws, int64_t E) {
  const int64_t r = (long_cap_rows(E) + 3) / 4 * 4, it = (long_cap_items(E) + 3) / 4 * 4;
  LongView v;
  v.cnt = ws;
  v.done = ws + 4;
  v.row = v.done + r;
  v.item0 = v.row + r;
  v.item_slot = v.item0 + r;
  v.partial = reinterpret_cast<float*>(v.item_slot + it);
  return v;
}
// fixed split of a hub row: nch chunks of lch edges (lch a multiple of the stage depth)
__host__ __device__ inline void long_chunking(int len, int& lch, int& nch) {
  int n0 = (len + LONG_ROW - 1) / LONG_ROW;
  if (n0 > LONG_MAX_CHUNKS) n0 = LONG_MAX_CHUNKS;
  if (n0 < 1) n0 = 1;
  lch = ((len + n0 - 1) / n0 + 7) / 8 * 8;
  if (lch < 8) lch = 8;
  nch = (len + lch - 1) / lch;
}

struct Csr {
  const int32_t* ptr;
  const int32_t* idx;
  int32_t* lng;   // hub-row list of this CSR or nullptr (rows are then walked by their owner)
  int64_t E;      // edge capacity the hub-row list was laid out for
};

// edge weights.  row(i) is read once per row; the self-loop term of row i is self(row(i)).
// GCN: w(e: j -> i) = dis[j] * dis[i], plus the self-loop dis[i]^2.
struct WtGcn {
  const float* dis;
  static constexpr bool kSelf = true;
  __device__ __forceinline__ float row(int i) const { return dis[i]; }
  __device__ __forceinline__ float edge(int, int j, float drow) const { return __fmul_rn(dis[j], drow); }
  __device__ __forceinline__ float self(float drow) const { return __fmul_rn(drow, drow); }
};
// edge-weighted GCN: the normalised weight of every CSR entry and of every self-loop, precomputed
// (weighted.cu, (dis[j] * w_e) * dis[i] as gcn_norm forms it) and read as they are
struct WtEntry {
  const float* val;    // [E] per CSR entry, in the order of the CSR being swept
  const float* slf;    // [N] per node
  static constexpr bool kSelf = true;
  __device__ __forceinline__ float row(int i) const { return slf[i]; }
  __device__ __forceinline__ float edge(int e, int, float) const { return val[e]; }
  __device__ __forceinline__ float self(float s) const { return s; }
};
// explicit per-entry weights, no self term (column-sorted X for the weight gradient)
struct WtVal {
  const float* val;
  static constexpr bool kSelf = false;
  __device__ __forceinline__ float row(int) const { return 0.f; }
  __device__ __forceinline__ float edge(int e, int, float) const { return val[e]; }
  __device__ __forceinline__ float self(float) const { return 0.f; }
};

// Post functors: operator()(row, sum, sub, half mask, scratch) finishes one row; kPairs = true
// adds pair(row, v0, ok0, v1, ok1, ...) for rows (row, row + 1) with two scratch rows; kInline = true: a light
// epilogue that needs no scratch row and is called as soon as a row's sum is complete (no trip through the stage).
// plain feature rows: val(j) = h[j, :]
struct ValRow {
  static constexpr bool kHasAux = false;
  const float* h;
  int64_t ldh;
  __device__ __forceinline__ void fetch(float* dst, int j, int sub) const {
    cp_async_row16(dst + 4 * sub, h + (int64_t)j * ldh + 4 * sub);
  }
  __device__ __forceinline__ int aux(int) const { return 0; }
  __device__ __forceinline__ float4 value(const float* slot, int, int sub) const { return ld4(slot + 4 * sub); }
};

// shared memory a sweep needs per CTA (256 threads = 16 half-warps).  Per half-warp:
//   stage[(R + Q)][64]  self rows (later: the finished row sums), neighbour rows of a round
//   sw[Q] weights, su[Q] row of each staged edge, sa[Q + R] per-row aux values,
//   sp[R + 1] CSR pointers, sq[R + 1] offsets in the block's edge stream, sd[R] dis of the rows
template <int R, int Q>
struct SweepSmem {
  static constexpr int kStageFloats = 16 * (R + Q) * H;
  static constexpr int kMetaInts = 3 * Q + 4 * R + 2;   // per half-warp
  static constexpr int kBytes = kStageFloats * 4 + 16 * kMetaInts * 4 + 16;
};

// units of 2*R rows per CTA chunk: small batches spread over all SMs, large ones amortise
static inline int sweep_cb(int64_t N, int R, int max_ctas) {
  const int64_t nunits = ceil_div(ceil_div(N, R), 2);
  int64_t cb = nunits / ((int64_t)max_ctas * 8);
  if (cb < 8) cb = 8;      // at least one unit per warp of the CTA
  if (cb > 16) cb = 16;
  return (int)cb;
}
static inline int sweep_grid(int64_t N, int R, int cb, int max_ctas) {
  int64_t blocks = ceil_div(ceil_div(ceil_div(N, R), 2), cb);
  if (blocks > max_ctas) blocks = max_ctas;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

template <int R, int Q, bool EXACT, class Wt, class Val, class Post>
__device__ __forceinline__ void csr_sweep(const Csr g, const Wt wt, const int n, const int cb, float* smem_dyn,
                                          const Val val, const Post post) {
  static_assert(R <= 15 && Q <= 16, "one lane per row pointer / staged edge");
  const int lane = threadIdx.x & 31, sub = lane & 15, half = lane >> 4;
  const int hw = threadIdx.x >> 4;
  const unsigned hm = half_mask(half);
  float* st = smem_dyn + (size_t)hw * (R + Q) * H;
  int* meta = reinterpret_cast<int*>(smem_dyn + SweepSmem<R, Q>::kStageFloats) + hw * SweepSmem<R, Q>::kMetaInts;
  float* sw = reinterpret_cast<float*>(meta);
  int* su = meta + Q;
  int* sa = meta + 2 * Q;            // [Q] neighbours, [R] own rows
  int* sp = meta + 3 * Q + R;        // [R + 1]
  int* sq = sp + R + 1;              // [R + 1]
  float* sd = reinterpret_cast<float*>(sq + R + 1);   // [R]
  int* s_next = reinterpret_cast<int*>(smem_dyn + SweepSmem<R, Q>::kStageFloats) + 16 * SweepSmem<R, Q>::kMetaInts;
  if (threadIdx.x == 0) *s_next = 0;
  __syncthreads();
  const int nblocks = (n + R - 1) / R;
  const int nunits = (nblocks + 1) / 2;
  for (;;) {
    __syncwarp();
    int t = 0;
    if (lane == 0) t = atomicAdd(s_next, 1);
    t = __shfl_sync(FULL_MASK, t, 0);
    const int64_t chunk = (int64_t)blockIdx.x + (int64_t)(t / cb) * gridDim.x;
    if (chunk * cb >= nunits) break;
    const int unit = (int)(chunk * cb) + t % cb;
    const int i0 = (unit * 2 + half) * R;
    const int nrows = max(0, min(R, n - i0));
    // row pointers, dis and aux of the block: one lane per row
    if (sub <= nrows && nrows > 0) sp[sub] = g.ptr[i0 + sub];
    if (sub < nrows) {
      sd[sub] = wt.row(i0 + sub);
      if constexpr (Wt::kSelf && Val::kHasAux) sa[Q + sub] = val.aux(i0 + sub);
    }
    if (Wt::kSelf) {
#pragma unroll
      for (int u = 0; u < R; ++u)
        if (u < nrows) val.fetch(st + u * H, i0 + u, sub);
    }
    __syncwarp();
    // offsets of the rows in the block's edge stream (a 16-lane prefix sum of the row lengths); hub rows are left
    // to the split path and take no room in the stream
    int len = 0;
    bool is_long = false;
    if (sub < nrows) {
      len = sp[sub + 1] - sp[sub];
      is_long = len > LONG_ROW && g.lng != nullptr;
      if (is_long) len = 0;
    }
    int inc = len;
#pragma unroll
    for (int o = 1; o < 16; o <<= 1) {
      const int t_up = __shfl_up_sync(FULL_MASK, inc, o, 16);
      if (sub >= o) inc += t_up;
    }
    const int ne = __shfl_sync(FULL_MASK, inc, 15, 16);
    if (sub <= R) sq[sub] = sub < nrows ? inc - len : ne;
    const unsigned longmask = (__ballot_sync(FULL_MASK, is_long) >> (half * 16)) & 0xffffu;
    __syncwarp();
    const int nemax = max(ne, __shfl_xor_sync(FULL_MASK, ne, 16));
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int cur = -1;              // row whose sum is being accumulated
    unsigned flushed = 0;      // rows whose finished sum sits in their stage slot
    // finished row: add the self-loop term and park the sum in the row's own stage slot
    auto flush = [&](int u) {
      if (Wt::kSelf) {
        acc_add<EXACT>(acc, wt.self(sd[u]), val.value(st + u * H, sa[Q + u], sub));
      }
      if constexpr (Post::kInline) post(i0 + u, acc, sub, hm, nullptr);   // light epilogue: finish the row right here
      else st4(st + u * H + 4 * sub, acc);
      flushed |= 1u << u;
    };
    for (int r0 = 0; r0 < nemax; r0 += Q) {
      const int nb = max(0, min(Q, ne - r0));
      const int nbmax = min(Q, nemax - r0);
      int j = 0;
      if (sub < nb) {
        const int s = r0 + sub;
        int u = 0;   // largest u with sq[u] <= s (sq is non-decreasing, sq[0] = 0): binary search over the R offsets
        if constexpr (R == 8) {
          u = s >= sq[4] ? 4 : 0;
          u += s >= sq[u + 2] ? 2 : 0;
          u += s >= sq[u + 1] ? 1 : 0;
        } else {
#pragma unroll
          for (int k = 1; k < R; ++k) u += (s >= sq[k]) ? 1 : 0;
        }
        const int e = sp[u] + (s - sq[u]);
        j = g.idx[e];
        sw[sub] = wt.edge(e, j, sd[u]);
        su[sub] = u;
        if constexpr (Val::kHasAux) sa[sub] = val.aux(j);
      }
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        if (q < nbmax) {
          const int jj = __shfl_sync(FULL_MASK, j, q, 16);
          if (q < nb) val.fetch(st + (R + q) * H, jj, sub);
        }
      }
      cp_async_commit_wait_all();
      __syncwarp();
#pragma unroll 2
      for (int q = 0; q < nb; ++q) {
        const int u = su[q];
        if (u != cur) {
          if (cur >= 0) flush(cur);
          cur = u;
          acc = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        acc_add<EXACT>(acc, sw[q], val.value(st + (R + q) * H, sa[q], sub));
      }
      __syncwarp();
    }
    cp_async_commit_wait_all();   // blocks without edges: the self rows are still in flight
    __syncwarp();
    if (cur >= 0) flush(cur);
    auto finished = [&](int u) {   // the row's sum (self-loop included)
      float4 v;
      if ((flushed >> u) & 1u) {
        v = ld4(st + u * H + 4 * sub);   // a lane re-reads only what it wrote itself
      } else {
        v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (Wt::kSelf) {
          acc_add<EXACT>(v, wt.self(sd[u]), val.value(st + u * H, sa[Q + u], sub));
        }
      }
      return v;
    };
    if constexpr (Post::kPairs) {   // epilogues that share work between two rows (one pass over W for both)
#pragma unroll 1
      for (int u = 0; u < nrows; u += 2) {
        const bool ok0 = !((longmask >> u) & 1u), ok1 = u + 1 < nrows && !((longmask >> (u + 1)) & 1u);
        if (!ok0 && !ok1) continue;
        const float4 v0 = ok0 ? finished(u) : make_float4(0.f, 0.f, 0.f, 0.f);
        const float4 v1 = ok1 ? finished(u + 1) : make_float4(0.f, 0.f, 0.f, 0.f);
        post.pair(i0 + u, v0, ok0, v1, ok1, sub, hm, st + R * H);
      }
    } else {
#pragma unroll 1
      for (int u = 0; u < nrows; ++u) {
        if ((longmask >> u) & 1u) continue;
        if (Post::kInline && ((flushed >> u) & 1u)) continue;   // posted when its last edge was added
        post(i0 + u, finished(u), sub, hm, st + (R + (u & (Q - 1))) * H);
      }
    }
  }
  // ---- hub rows: items (row, chunk) spread over all half-warps of the grid --------------------
  if (g.lng == nullptr) return;
  const LongView L = long_view(g.lng, g.E);
  const int n_items = L.cnt[1];
  for (int t = blockIdx.x * 16 + hw; t < n_items; t += gridDim.x * 16) {
    const int slot = L.item_slot[t];
    const int row = L.row[slot];
    const int item0 = L.item0[slot];
    const int rs = g.ptr[row], len = g.ptr[row + 1] - rs;
    int lch, nch;
    long_chunking(len, lch, nch);
    const int s = rs + (t - item0) * lch, e = min(rs + len, s + lch);
    const float d = wt.row(row);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int e0 = s; e0 < e; e0 += Q) {
      const int nb = min(Q, e - e0);
      int j = 0;
      if (sub < nb) {
        j = g.idx[e0 + sub];
        sw[sub] = wt.edge(e0 + sub, j, d);
        sa[sub] = val.aux(j);
      }
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        const int jj = __shfl_sync(hm, j, q, 16);
        if (q < nb) val.fetch(st + (R + q) * H, jj, sub);
      }
      cp_async_commit_wait_all();
      __syncwarp(hm);
      for (int q = 0; q < nb; ++q) acc_add<EXACT>(acc, sw[q], val.value(st + (R + q) * H, sa[q], sub));
      __syncwarp(hm);
    }
    __stcg(reinterpret_cast<float4*>(L.partial + (size_t)t * H + 4 * sub), acc);
    __threadfence();
    __syncwarp(hm);
    int old = 0;
    if (sub == 0) old = atomicAdd(&L.done[slot], 1);
    old = __shfl_sync(hm, old, 0, 16);
    if (old == nch - 1) {   // last chunk in: ordered combine, self-loop, epilogue
      __threadfence();
      if (Wt::kSelf) {
        val.fetch(st, row, sub);
        if (sub == 0) sa[Q] = val.aux(row);
      }
      float4 tot = make_float4(0.f, 0.f, 0.f, 0.f);
      const float* p0 = L.partial + (size_t)item0 * H + 4 * sub;
      for (int c0 = 0; c0 < nch; c0 += 8) {   // eight partials in flight, added in chunk order
        float4 pv[8];
#pragma unroll
        for (int u = 0; u < 8; ++u)
          pv[u] = c0 + u < nch ? __ldcg(reinterpret_cast<const float4*>(p0 + (size_t)(c0 + u) * H))
                               : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          if (c0 + u < nch) {
            tot.x = __fadd_rn(tot.x, pv[u].x);
            tot.y = __fadd_rn(tot.y, pv[u].y);
            tot.z = __fadd_rn(tot.z, pv[u].z);
            tot.w = __fadd_rn(tot.w, pv[u].w);
          }
        }
      }
      cp_async_commit_wait_all();
      __syncwarp(hm);
      if (Wt::kSelf) acc_add<EXACT>(tot, wt.self(d), val.value(st, sa[Q], sub));
      if (sub == 0) L.done[slot] = 0;   // ready for the next launch over this CSR
      post(row, tot, sub, hm, st + R * H);
    }
    __syncwarp(hm);
  }
}

}  // namespace bigcn
