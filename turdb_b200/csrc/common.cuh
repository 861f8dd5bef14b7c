// common.cuh — shared device helpers for libturdb_cuda (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace turdb {

constexpr uint32_t kInvalid = 0xFFFFFFFFu;
constexpr uint32_t kExpandedBit = 0x80000000u;  // bit 31 of a list id: adjacency already read
constexpr uint32_t kFullMask = 0xFFFFFFFFu;
constexpr uint32_t kL0 = 32;  // MAX_L0_NEIGHBORS, src/hnsw/mod.rs:126
constexpr uint32_t kUp = 16;  // MAX_LEVEL_NEIGHBORS, src/hnsw/mod.rs:127

enum Metric : int { kL2 = 0, kCosine = 1, kIP = 2 };

// Device view of the uploaded index (DESIGN.md §3).
struct DeviceIndex {
  const float* arena;       // [n][ds] row stride ds = round_up(dim, 4) floats, 16 B aligned rows
  const float* norm2;       // [n] dot(b, b) in the reference's AVX2 lane order (cosine only)
  const uint32_t* l0_adj;   // [n][32], INVALID padded
  const uint32_t* up_base;  // [n]
  const uint32_t* up_adj;   // [slots][16], INVALID padded
  const uint64_t* row_ids;  // [n]
  const uint8_t* levels;    // [n]
  uint64_t n;
  uint32_t dim;
  uint32_t ds;
  uint32_t entry;
  uint32_t max_level;
  // rows still in the table (turdb_cuda_index_delete): bit i of word i / 64; null until the first delete = every row.
  // The traversal never reads it (the launch hands it over as the visibility bitmap); the exact / SQL kernels do.
  const uint64_t* live;
};

__device__ __forceinline__ bool node_live(const DeviceIndex& ix, uint32_t id) {
  return !ix.live || ((ix.live[id >> 6] >> (id & 63)) & 1ull) != 0;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier + TMA bulk copy (cp.async.bulk; SASS: UBLKCP) ---------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// global -> shared bulk copy, completion counted in bytes on `bar`.  16 B aligned, size % 16 == 0.
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
      "l"(src), "r"(bytes), "r"(bar)
      : "memory");
}

// L2 prefetch of a byte range (cp.async.bulk.prefetch.L2; 16 B aligned, size % 16 == 0): no destination, no barrier.
__device__ __forceinline__ void bulk_prefetch_l2(const void* src, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}

// ---- the reference's AVX2 reduction order, one QUAD (4 lanes) per vector ---------------------
// Lane p of a quad owns AVX lanes 2p and 2p+1 (distance.rs:105-129): it walks elements 8t+2p,
// 8t+2p+1 with one fused multiply-add each, then the quad reproduces horizontal_sum_avx2
// (distance.rs:150-161): (lo128 + hi128) = xor-2 exchange, movehl add = xor-1 exchange, x + y.
__device__ __forceinline__ float quad_hsum(float2 acc) {
  acc.x = __fadd_rn(acc.x, __shfl_xor_sync(kFullMask, acc.x, 2));
  acc.y = __fadd_rn(acc.y, __shfl_xor_sync(kFullMask, acc.y, 2));
  acc.x = __fadd_rn(acc.x, __shfl_xor_sync(kFullMask, acc.x, 1));
  acc.y = __fadd_rn(acc.y, __shfl_xor_sync(kFullMask, acc.y, 1));
  return __fadd_rn(acc.x, acc.y);
}

// Packed FP32x2 math (Blackwell FADD2 / FFMA2): both halves are IEEE round-to-nearest, so each AVX
// lane's chain is bit-identical to the scalar fmaf chain.
__device__ __forceinline__ uint64_t sub2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ float2 unpack2(uint64_t v) {
  float2 f;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(f.x), "=f"(f.y) : "l"(v));
  return f;
}

// Accumulate `nsteps` AVX steps (8 elements each) of a quad's chain.  av/bv already point at this lane's
// float2 of the first step (base + 8*step0 + 2p floats); consecutive steps are 4 uint64 apart.
template <bool L2>
__device__ __forceinline__ uint64_t quad_accum(uint64_t acc, const uint64_t* av, const uint64_t* bv, uint32_t nsteps) {
  uint32_t t = 0;
  for (; t + 8 <= nsteps; t += 8, av += 32, bv += 32) {
    uint64_t x[8], y[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      x[u] = av[4 * u];
      y[u] = bv[4 * u];
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      if (L2) {
        const uint64_t d = sub2(x[u], y[u]);
        acc = fma2(d, d, acc);
      } else {
        acc = fma2(x[u], y[u], acc);
      }
    }
  }
  for (; t < nsteps; ++t, av += 4, bv += 4) {
    if (L2) {
      const uint64_t d = sub2(av[0], bv[0]);
      acc = fma2(d, d, acc);
    } else {
      acc = fma2(av[0], bv[0], acc);
    }
  }
  return acc;
}

// horizontal sum + the unfused scalar tail (distance.rs:120-126 / 225-229); a_tail/b_tail point at element 8*steps
template <bool L2>
__device__ __forceinline__ float quad_finish(uint64_t acc, const float* a_tail, const float* b_tail, uint32_t ntail) {
  float r = quad_hsum(unpack2(acc));
  for (uint32_t i = 0; i < ntail; ++i) {
    if (L2) {
      const float d = __fsub_rn(a_tail[i], b_tail[i]);
      r = __fadd_rn(r, __fmul_rn(d, d));
    } else {
      r = __fadd_rn(r, __fmul_rn(a_tail[i], b_tail[i]));
    }
  }
  return r;
}

// a, b: 8 B aligned float pointers (shared or global); p = lane & 3.  Returns squared L2.
__device__ __forceinline__ float quad_l2sq(const float* a, const float* b, uint32_t dim, uint32_t p) {
  const uint32_t steps = dim >> 3;
  const uint64_t acc = quad_accum<true>(0ull, reinterpret_cast<const uint64_t*>(a) + p,
                                        reinterpret_cast<const uint64_t*>(b) + p, steps);
  return quad_finish<true>(acc, a + (steps << 3), b + (steps << 3), dim & 7);
}

__device__ __forceinline__ float quad_dot(const float* a, const float* b, uint32_t dim, uint32_t p) {
  const uint32_t steps = dim >> 3;
  const uint64_t acc = quad_accum<false>(0ull, reinterpret_cast<const uint64_t*>(a) + p,
                                         reinterpret_cast<const uint64_t*>(b) + p, steps);
  return quad_finish<false>(acc, a + (steps << 3), b + (steps << 3), dim & 7);
}

// ---- SQ8 rows (SQ8Vector, src/hnsw/quantization.rs:60-116): dim u8 codes | pad to 4 | min f32 | scale f32 ----
// A quad walks the codes in the same AVX2 lane order as the FP32 rows; every element is decoded exactly as
// SQ8Vector::decode does (min + (q as f32) * scale, two roundings, quantization.rs:108-113) before it enters the
// chain, so the value equals the FP32 functions applied to the decoded vector bit for bit.
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ uint64_t pack2(float x, float y) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(x), "f"(y));
  return r;
}
// Two codes -> two decoded floats.  `q as f32` without the conversion pipe: 0x4B000000 | q is the float 2^23 + q,
// and subtracting 2^23 is exact; then the reference's two roundings, q * scale and min + (.), as packed FP32x2.
__device__ __forceinline__ uint64_t sq8_pair(const uint8_t* row, uint32_t step, uint32_t p, uint64_t mn2, uint64_t sc2) {
  const uint2 w = *reinterpret_cast<const uint2*>(row + 8 * step);  // the 8 codes of this AVX step (quad broadcast)
  const uint32_t word = (p & 2) ? w.y : w.x;
  // byte_perm over {word (bytes 0-3), 0x4B000000 (bytes 4-7)}: result = 4B 00 00 cc
  const uint32_t sel0 = 0x7440u | (2 * (p & 1)), sel1 = sel0 | 1u;
  const float f0 = __uint_as_float(__byte_perm(word, 0x4B000000u, sel0));
  const float f1 = __uint_as_float(__byte_perm(word, 0x4B000000u, sel1));
  // ptxas 12.9 contracts mul.rn.f32x2 + add.rn.f32x2 into one FFMA2 (seen in SASS; one rounding instead of the
  // reference's two), so the products are formed by scalar FMULs, which it leaves alone
  const float2 q = unpack2(add2(pack2(f0, f1), pack2(-8388608.0f, -8388608.0f)));
  const float2 sc = unpack2(sc2);
  return add2(mn2, pack2(__fmul_rn(q.x, sc.x), __fmul_rn(q.y, sc.y)));
}
// MODE 0: squared L2 of (a, decode(row)); 1: dot(a, decode(row)); 2: dot(decode(row), decode(row)) (a unused)
template <int MODE>
__device__ __forceinline__ float quad_sq8(const float* a, const uint8_t* row, uint32_t dim, uint32_t p) {
  const uint32_t steps = dim >> 3, tail0 = steps << 3;
  const float* ms = reinterpret_cast<const float*>(row + ((dim + 3) & ~3u));
  const float mn = ms[0], sc = ms[1];
  const uint64_t mn2 = pack2(mn, mn), sc2 = pack2(sc, sc);
  const uint64_t* av = reinterpret_cast<const uint64_t*>(a) + p;
  uint64_t acc = 0ull;
#pragma unroll 4
  for (uint32_t t = 0; t < steps; ++t) {
    const uint64_t b = sq8_pair(row, t, p, mn2, sc2);
    if (MODE == 0) {
      const uint64_t d = sub2(av[4 * t], b);
      acc = fma2(d, d, acc);
    } else if (MODE == 1) {
      acc = fma2(av[4 * t], b, acc);
    } else {
      acc = fma2(b, b, acc);
    }
  }
  float r = quad_hsum(unpack2(acc));
  for (uint32_t i = tail0; i < dim; ++i) {  // the unfused scalar tail (distance.rs:120-126 / 225-229)
    const float b = __fadd_rn(mn, __fmul_rn((float)row[i], sc));
    if (MODE == 0) {
      const float d = __fsub_rn(a[i], b);
      r = __fadd_rn(r, __fmul_rn(d, d));
    } else if (MODE == 1) {
      r = __fadd_rn(r, __fmul_rn(a[i], b));
    } else {
      r = __fadd_rn(r, __fmul_rn(b, b));
    }
  }
  return r;
}

// cosine_avx2's epilogue, distance.rs:279-284
__device__ __forceinline__ float cosine_finish(float dot, float na, float nb) {
  float np = __fsqrt_rn(__fmul_rn(na, nb));
  if (np == 0.0f) return 1.0f;
  return __fsub_rn(1.0f, __fdiv_rn(dot, np));
}

}  // namespace turdb
