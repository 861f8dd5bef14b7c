// exact_search.cuh — the exact (brute-force) path and the multi-shard top-k merge.
//
// Exact path = the SQL `ORDER BY vec <op> q LIMIT k` scan (TopKExec, src/sql/executor.rs:2239-2392) as
//   (1) a BF16 tensor-core pass  S = Q · X^T  (tcgen05.mma, accumulators in TMEM, operands staged by TMA),
//       whose epilogue turns each score into a ranking key (key = s * a[col] + b[col]; larger = closer) and
//       keeps only keys above the query's running threshold (rare) in a per-query candidate buffer;
//   (2) a threshold update between passes over geometrically growing slices of the corpus
//       (k' = rerank_factor * k best keys so far -> new threshold);
//   (3) an FP32 rerank of the k' survivors in the reference's AVX2 lane order (bit-identical to
//       select_squared_distance_fn, src/hnsw/distance.rs:438-444) and the final ascending top-k.
// The dense contraction is the only tensor-core use in this library.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace turdb {

// ------------------------------------------------------------------------------------------------
// shard merge
// ------------------------------------------------------------------------------------------------
// One warp per query: k-way merge of n_shards ascending lists; at every step the head with the smallest
// (distance, row_id, shard) wins.  gathered_* are [n_shards][nq][k]; lane s walks shard s (n_shards <= 32).
// Shard s's arrays start s * stride bytes after the base pointers (dense [n_shards][nq][k] arrays: stride = the array's
// size; one packed block per shard, as a single all-gather delivers it: stride = the block's size for all three).
__global__ void merge_topk_kernel(const uint8_t* __restrict__ g_rows_b, const uint8_t* __restrict__ g_dist_b,
                                  const uint8_t* __restrict__ g_counts_b, size_t rows_stride, size_t dist_stride,
                                  size_t cnt_stride, uint32_t n_shards, uint32_t nq,
                                  uint32_t k, uint64_t* __restrict__ out_rows, float* __restrict__ out_dist,
                                  uint32_t* __restrict__ out_counts) {
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (q >= nq) return;
  uint32_t head = 0, cnt = 0;
  const size_t base = (size_t)q * k;
  const uint64_t* g_rows = nullptr;
  const float* g_dist = nullptr;
  if (lane < n_shards) {
    g_rows = reinterpret_cast<const uint64_t*>(g_rows_b + lane * rows_stride);
    g_dist = reinterpret_cast<const float*>(g_dist_b + lane * dist_stride);
    cnt = min(reinterpret_cast<const uint32_t*>(g_counts_b + lane * cnt_stride)[q], k);
  }
  uint32_t produced = 0;
  for (; produced < k; ++produced) {
    float d = INFINITY;
    uint64_t r = 0xFFFFFFFFFFFFFFFFull;
    bool have = head < cnt;
    if (have) {
      d = g_dist[base + head];
      r = g_rows[base + head];
    }
    if (!__any_sync(kFullMask, have)) break;
    float bd = d;
    uint64_t br = r;
    uint32_t bl = have ? lane : 0xFFFFFFFFu;
#pragma unroll
    for (uint32_t off = 16; off >= 1; off >>= 1) {
      float od = __shfl_xor_sync(kFullMask, bd, off);
      uint64_t orow = __shfl_xor_sync(kFullMask, br, off);
      uint32_t ol = __shfl_xor_sync(kFullMask, bl, off);
      bool take = (ol != 0xFFFFFFFFu) && (bl == 0xFFFFFFFFu || od < bd || (od == bd && orow < br) ||
                                          (od == bd && orow == br && ol < bl));
      if (take) {
        bd = od;
        br = orow;
        bl = ol;
      }
    }
    if (lane == bl) head += 1;
    if (lane == 0) {
      out_rows[(size_t)q * k + produced] = br;
      out_dist[(size_t)q * k + produced] = bd;
    }
  }
  for (uint32_t i = produced + lane; i < k; i += 32) {
    out_rows[(size_t)q * k + i] = 0xFFFFFFFFFFFFFFFFull;
    out_dist[(size_t)q * k + i] = INFINITY;
  }
  if (lane == 0) out_counts[q] = produced;
}

// ------------------------------------------------------------------------------------------------
// operand preparation
// ------------------------------------------------------------------------------------------------
// 16-bit operand formats of the filter (tcgen05 kind::f16 takes either): BF16 (8-bit mantissa, FP32 range) or FP16 (11-bit
// mantissa — an 8x smaller rounding error, hence an 8x narrower slack band and far fewer rows to rerank — but values
// beyond +-65504 overflow).  The arena copy is FP16 whenever its largest |value| allows (always for the cosine copy, whose
// rows are pre-scaled to unit length), else BF16; queries are converted to the arena copy's format per call, and a
// query that overflows it gets an infinite error bound and is served by the streaming scan.
__device__ __forceinline__ uint16_t to_half_bits(float v, int fp16) {
  return fp16 ? __half_as_ushort(__float2half_rn(v)) : __bfloat16_as_ushort(__float2bfloat16_rn(v));
}
__device__ __forceinline__ float from_half_bits(uint16_t b, int fp16) {
  return fp16 ? __half2float(__ushort_as_half(b)) : __bfloat162float(__ushort_as_bfloat16(b));
}

// FP32 rows [rows][ds] -> 16-bit rows [rows][kp] (kp = dim rounded up to 64, zero padded).  With `norm2` the row is
// scaled by 1/|x| first, so that the cosine pass's score q.x/|x| is already its ranking key.
// `aug` fills columns dim, dim+1, dim+2 (the L2 form: the contraction itself produces key = q.x - |x|^2/2):
//   1 (vector side): the 16-bit hi / mid / lo split of t = -norm2[r] / (2 * aug_scale) — h1 = rn16(t), h2 = rn16(t - h1),
//     h3 = rn16(t - h1 - h2); the differences are exact in FP32, so aug_scale * (h1 + h2 + h3) misses -|x|^2/2 by less than
//     2^-23 of it (three 8-bit BF16 mantissas) plus, in FP16, aug_scale * 2^-24 (subnormal spacing);
//   2 (query side): aug_scale in each of the three columns (a power of two: exact in either format).
// With aug == 1 `norm2` is NOT a scaling (rows stay raw).
__global__ void to_half_kernel(const float* __restrict__ src, uint32_t dim, uint32_t ds, uint32_t kp,
                               uint64_t rows, const float* __restrict__ norm2, int fp16, uint16_t* __restrict__ dst, int aug = 0,
                               float aug_scale = 1.f) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * kp) return;
  const uint64_t r = i / kp;
  const uint32_t c = (uint32_t)(i % kp);
  float v = c < dim ? src[r * ds + c] : 0.f;
  if (aug == 0 && norm2) {
    const float n2 = norm2[r];
    v = n2 > 0.f ? v * rsqrtf(n2) : 0.f;
  }
  if (aug == 2 && c >= dim && c < dim + 3) v = aug_scale;
  if (aug == 1 && c >= dim && c < dim + 3) {
    const float t = -0.5f * norm2[r] / aug_scale;  // aug_scale is a power of two: exact
    const float h1 = from_half_bits(to_half_bits(t, fp16), fp16);
    const float h2 = from_half_bits(to_half_bits(t - h1, fp16), fp16);
    v = c == dim ? h1 : (c == dim + 1 ? h2 : (t - h1) - h2);
  }
  dst[i] = to_half_bits(v, fp16);
}

// largest value of a non-negative float array (bit patterns order like the values)
__global__ void max_nonneg_kernel(const float* __restrict__ src, uint64_t n, uint32_t* __restrict__ out) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float m = i < n ? src[i] : 0.f;
  if (!(m >= 0.f)) m = 0.f;
  for (uint32_t off = 16; off >= 1; off >>= 1) m = fmaxf(m, __shfl_xor_sync(kFullMask, m, off));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(out, __float_as_uint(m));
}

// largest |value| of the arena (picks the copy's format)
__global__ void max_abs_kernel(const float* __restrict__ src, uint32_t dim, uint32_t ds, uint64_t rows, uint32_t* __restrict__ out) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float m = 0.f;
  if (i < rows * dim) m = fabsf(src[(i / dim) * ds + (i % dim)]);
  for (uint32_t off = 16; off >= 1; off >>= 1) m = fmaxf(m, __shfl_xor_sync(kFullMask, m, off));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(out, __float_as_uint(m));
}

// What the BF16 rounding cost, per operand set: max over rows of |v - bf16(v)|_2 and of |bf16(v)|_2 (v = the FP32 row
// that was converted: raw, or scaled by 1/|x| for the cosine copy).  One warp per row; the maxima are kept as the bit
// patterns of non-negative floats (atomicMax on uint32).  They bound the filter's score error (query_slack_kernel), so
// that the tensor-core pass is a CERTIFIED filter: it never drops a row the exact ranking would keep.
__global__ void bf16_rowerr_kernel(const float* __restrict__ src, uint32_t dim, uint32_t ds, uint32_t kp, uint64_t rows,
                                   const float* __restrict__ norm2, const uint16_t* __restrict__ conv, int fp16,
                                   uint32_t* __restrict__ out_max2) {
  const uint64_t r = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = threadIdx.x & 31;
  if (r >= rows) return;
  float sc = 1.f;
  if (norm2) {
    const float n2 = norm2[r];
    sc = n2 > 0.f ? rsqrtf(n2) : 0.f;
  }
  float e2 = 0.f, n2b = 0.f;
  for (uint32_t c = lane; c < dim; c += 32) {
    const float v = src[r * ds + c] * sc, b = from_half_bits(conv[r * kp + c], fp16);
    e2 = fmaf(v - b, v - b, e2);
    n2b = fmaf(b, b, n2b);
  }
  for (uint32_t off = 16; off >= 1; off >>= 1) {
    e2 += __shfl_xor_sync(kFullMask, e2, off);
    n2b += __shfl_xor_sync(kFullMask, n2b, off);
  }
  if (lane == 0) {
    atomicMax(out_max2 + 0, __float_as_uint(sqrtf(e2) * 1.0001f));
    atomicMax(out_max2 + 1, __float_as_uint(sqrtf(n2b) * 1.0001f));
  }
}

// Per query: 2 e(q), where e(q) bounds |filter key - exact key| for EVERY row of the corpus (key as defined below,
// larger = closer).  With q~, x~ the BF16-rounded operands, dq = |q - q~|, Dx = max |x - x~|, Xn = max |x~|:
//   |q~.x~ - q.x| <= |q| Dx + dq Xn                       (rounding of the operands)
//                  + kp 2^-22 (|q| + dq) Xn               (FP32 accumulation inside the tensor core, generous)
//   + FP32 evaluation of the bias / of the value the exact ranking uses (AVX2-order FP32 or the SQL operator's f64 of
//     f32 differences): 2^-22 (dim/8 + 8) (|q| + Xn + Dx)^2 for L2, 2^-20 |q| for the pre-scaled cosine rows.
// The filter admits a key >= tau - 2 e(q) where tau is the kprime-th best FILTER key seen so far; a rejected row then
// has an exact key below the exact keys of kprime admitted rows.
// `aug_scale` > 0: the L2 bias travels inside the contraction (three extra columns, see to_half_kernel): its split
// residual (2^-23 bmax + aug_scale 2^-24) and the FP32 accumulation over the three extra products (kp 2^-22 bmax, with
// bmax = (Xn + Dx)^2 / 2 >= max |x|^2 / 2) join the bound.
__global__ void query_slack_kernel(const float* __restrict__ queries, uint32_t dim, uint32_t kp, uint32_t nq,
                                   const uint16_t* __restrict__ qconv, int fp16, const uint32_t* __restrict__ arena_max2,
                                   int metric, float scale, float* __restrict__ slack, float aug_scale = 0.f) {
  const uint32_t q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (q >= nq) return;
  float e2 = 0.f, n2 = 0.f;
  for (uint32_t c = lane; c < dim; c += 32) {
    const float v = queries[(size_t)q * dim + c], b = from_half_bits(qconv[(size_t)q * kp + c], fp16);
    e2 = fmaf(v - b, v - b, e2);
    n2 = fmaf(v, v, n2);
  }
  for (uint32_t off = 16; off >= 1; off >>= 1) {
    e2 += __shfl_xor_sync(kFullMask, e2, off);
    n2 += __shfl_xor_sync(kFullMask, n2, off);
  }
  if (lane == 0) {
    const float dq = sqrtf(e2) * 1.0001f, qn = sqrtf(n2) * 1.0001f;
    const float Dx = __uint_as_float(arena_max2[0]), Xn = __uint_as_float(arena_max2[1]);
    float e = qn * Dx + dq * Xn + (float)kp * 2.3841858e-7f * (qn + dq) * Xn;
    if (metric == kL2) {
      const float s = qn + Xn + Dx;
      e += 2.3841858e-7f * (float)(dim / 8 + 8) * s * s;
      if (aug_scale > 0.f) {
        const float bmax = 0.5f * (Xn + Dx) * (Xn + Dx);
        e += 1.1920929e-7f * bmax + aug_scale * 5.9604645e-8f * 3.f + (float)kp * 2.3841858e-7f * bmax;
      }
    } else if (metric == kCosine) {
      e += 9.5367432e-7f * qn;
    } else {
      e += 2.3841858e-7f * (float)(dim / 8 + 8) * qn * (Xn + Dx);
    }
    slack[q] = 2.02f * e * scale;  // scale == 1 always, except under the TURDB_EXACT_SLACK_SCALE diagnostic (uncertified)
  }
}

// Fixed threshold of the range form (turdb_cuda_sql_range_batch, DESIGN §4.6): per statement, a filter key below which no
// row can satisfy `v <cmp> radius[q]`, v = the f32 projected value (sql_projection).  Only the near direction exists
// (v <= r for L2 / cosine, v >= r for IP), and `<` is treated as `<=` (a superset).  In f64, rounded toward admitting:
//   e  = slack[q] / 2 = 1.01 e(q) >= |filter key - real key|                  (query_slack_kernel)
//   g  = gamma_n = n u / (1 - n u), u = 2^-24: the bound of a sequential f32 sum of n rounded products, relative to
//        the sum of the absolute products
//   L2 : v = fl(sqrt(fl(sum fl(fl(q_i - x_i)^2)))) >= |q - x| (1 - u) sqrt(1 - gamma_{n+2}), so v <= r implies
//        |q - x| <= R = r / ((1 - u) sqrt(1 - gamma_{n+2})) and the key q.x - |x|^2/2 = (|q|^2 - |q - x|^2) / 2
//        >= (|q|^2 - R^2) / 2;                                         tau = (|q|^2 - R^2) / 2 - e
//   cos: the three f32 sums, two sqrts, product, quotient and 1 - . give |v - (1 - cos)| <= Ec (below), so v <= r
//        implies cos >= 1 - r - Ec; the key is |q| cos up to the rows' f32 scaling by rsqrtf(norm2) (relative
//        g + 4u, norm2 is itself an f32 sum);                          tau = |q| (1 - r - Ec) - |q| (g + 4u) - e
//   IP : |v - q.x| <= g |q| max|x|, max|x| <= Xn + Dx (arena_max2);   tau = r - g |q| (Xn + Dx) - e
// and every tau is lowered by 2^-30 of its terms' magnitudes (the f64 arithmetic here) and rounded down to f32.  A NaN
// radius compares false for every row (tau = +inf), a zero query under cosine is NULL for every row (+inf), and a
// bound that is not finite (a query overflowing the FP16 copy, an arena with +inf rows) admits every row (tau = -inf).
__global__ void range_thresh_kernel(const float* __restrict__ queries, uint32_t dim, uint32_t nq, int metric,
                                    const double* __restrict__ radius, const float* __restrict__ slack,
                                    const uint32_t* __restrict__ arena_max2, float* __restrict__ thresh) {
  const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  double qq = 0.0;  // |q|^2: every product is exact in f64, the sum is off by at most dim 2^-53 of it
  for (uint32_t i = 0; i < dim; ++i) {
    const double v = (double)queries[(size_t)q * dim + i];
    qq = fma(v, v, qq);
  }
  const double u = 0x1p-24, r = radius[q], e = 0.5 * (double)slack[q], qn = sqrt(qq);
  const double g = dim * u / (1.0 - dim * u);
  double t, mag;
  if (r != r) {
    t = INFINITY;
    mag = 0.0;
  } else if (metric == kL2) {
    const double g2 = (dim + 2) * u / (1.0 - (dim + 2) * u);
    const double R = fmax(r, 0.0) / ((1.0 - u) * sqrt(1.0 - g2));
    t = 0.5 * (qq - R * R) - e;
    mag = qq + R * R + e;
  } else if (metric == kCosine) {
    if (qq == 0.0) {
      t = INFINITY;
      mag = 0.0;
    } else {
      const double a = g + u;                                   // |n1 / |x| - 1|, |n2 / |q| - 1|
      const double B = (1.0 + a) * (1.0 + a) * (1.0 + u) - 1.0;  // |fl(n1 n2) / (|x||q|) - 1|
      const double Ec = ((u + B) + g * (1.0 + u)) / (1.0 - B) + 3.0 * u;
      t = qn * (1.0 - r - Ec) - qn * (g + 4.0 * u) - e;
      mag = qn * (1.0 + fabs(r) + Ec) + e;
    }
  } else {
    const double X = (double)__uint_as_float(arena_max2[0]) + (double)__uint_as_float(arena_max2[1]);
    t = r - g * qn * X - e;
    mag = fabs(r) + g * qn * X + e;
  }
  t -= 0x1p-30 * mag;
  if (t != t) t = -INFINITY;
  thresh[q] = __double2float_rd(t);
}

// Ranking key of a score for column (vector) j, larger = closer (the query's own norm does not change ranks) — in every
// case what the contraction itself produces:  L2: q.x - |x|^2/2 (three augmented columns of the L2 copy, to_half_kernel)
// cosine: q.x on rows pre-scaled by 1/|x|      IP: q.x

// ------------------------------------------------------------------------------------------------
// tcgen05 helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int32_t c0, int32_t c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, BF16 inputs, FP32 accumulate, M = 128
__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// K-major, 128-byte swizzle, 8-row groups 1024 B apart (cute::UMMA::SmemDescriptor, version 1 = Blackwell)
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);  // start address
  d |= (uint64_t)1 << 16;                      // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;            // stride byte offset
  d |= (uint64_t)1 << 46;                      // descriptor version
  d |= (uint64_t)2 << 61;                      // SWIZZLE_128B
  return d;
}
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void tmem_ld_32x32b_x32_nowait(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}

// ------------------------------------------------------------------------------------------------
// pass (1): GEMM + threshold filter
// ------------------------------------------------------------------------------------------------
// 256-column tiles: one MMA instruction covers N = 256, which halves the A bytes read from shared memory per flop.
//
// (r02, second half) What bounded this kernel was never the tensor pipe: 10k x 1M took 14 ms at 128-d, 13.5 ms at 384-d
// and 16.3 ms at 768-d, i.e. the time followed the number of SCORES, not the flops — the MMA issuer sat waiting for a
// drained accumulator (7.2k cycles per 128-d tile in the per-role cycle counters).  The epilogue is therefore built for
// latency, not for instruction count:
//  * sixteen epilogue warps (one per TMEM lane quarter x 64-column slice; TURDB_EXACT_EPI_COLS) so that four warps per
//    scheduler hide each other's dependent chains;
//  * per 32-column block: four 8-column group maxima and their maximum (3-input FMNMX), ONE warp vote; a block nobody's
//    threshold reaches costs ~25 instructions;
//  * a block that is reached looks only at the 8-column groups that are (one vote each), column by column with a ballot:
//    control flow stays warp-uniform, and the rare survivors go to a per-WARP queue in shared memory
//    (slot = running count + popc(ballot below me));
//  * when the queue passes 32 entries the whole warp flushes it: lane i reserves a slot in entry i's query buffer with
//    its own atomicAdd — one round trip for up to 64 candidates instead of one per thread.
//
// Two-CTA form (`PAIR`, tcgen05 cta_group::2): at K >= 384 the next bound is L2 -> SM bandwidth — 148 CTAs each streaming
// the whole slice need 148 x 192 KB per 256-column tile against ~6.3 KB/clk of L2 throughput = 4.6k cycles, above the
// 3.1k cycles of its MMAs.  A CTA pair (cluster of 2 on one TPC) shares every vector tile: each CTA stages HALF of the
// tile's rows (128 x 64 elements = 16 KB per stage) plus its own 128 queries, the leader issues M = 256 x N = 256 MMAs
// that read A from both CTAs and B halves from both, and each CTA's TMEM receives its own 128 query rows x 256 columns.
// L2 traffic and shared-memory fill per flop halve, and the B pipeline is twice as deep in time at the same bytes.
// Barriers: TMA of both CTAs completes on the LEADER's full barriers (.cta_group::2 form, leader arms 2x the bytes);
// tcgen05.commit multicasts "stage free" / "accumulator full" to both CTAs; both CTAs' epilogue warps arrive remotely on
// the leader's "accumulator drained" barrier.
#ifndef TURDB_EXACT_TILE_N
#define TURDB_EXACT_TILE_N 256
#endif
#ifndef TURDB_EXACT_EPI_COLS
#define TURDB_EXACT_EPI_COLS 64
#endif
constexpr uint32_t kTileM = 128;   // queries per CTA tile (UMMA M per CTA)
constexpr uint32_t kTileN = TURDB_EXACT_TILE_N;   // vectors per MMA tile (UMMA N): 128 or 256
constexpr uint32_t kChunkK = 64;   // 16-bit elements per 128 B swizzle row
constexpr uint32_t kChunkBytes = kTileM * kChunkK * 2;   // 16 KB per A (query) chunk
constexpr uint32_t kMaxStages = 8; // B pipeline depth is chosen at launch (as many stages as fit)
constexpr uint32_t kEpiCols = TURDB_EXACT_EPI_COLS;      // tile columns one epilogue warp owns
constexpr uint32_t kEpiWarps = 4 * (kTileN / kEpiCols);  // one per (TMEM lane quarter, column slice)
constexpr uint32_t kEpiThreads = 32 * kEpiWarps;
constexpr uint32_t kExactThreads = 64 + kEpiThreads;  // warp 0 TMA, warp 1 MMA + TMEM alloc, then the epilogue warps
constexpr uint32_t kWq = 64;       // entries of a warp's candidate queue (flushed when more than 32 are pending)
static_assert(kTileN == 128 || kTileN == 256, "UMMA N");
static_assert(kEpiCols == 32 || kEpiCols == 64 || kEpiCols == 128, "epilogue slice");
static_assert(kExactThreads <= 1024, "CTA size");

// bytes of one B (vector) chunk a CTA stages: the whole tile's rows, or half of them in the two-CTA form
__host__ __device__ constexpr uint32_t exact_b_chunk_bytes(bool pair, uint32_t tile_n) { return (pair ? tile_n / 2 : tile_n) * kChunkK * 2; }
__host__ __device__ constexpr uint32_t exact_stage_bytes(bool stream_a, bool pair, uint32_t tile_n) {
  return (stream_a ? kChunkBytes : 0u) + exact_b_chunk_bytes(pair, tile_n);
}
// everything in dynamic shared memory except the pipeline stages (kernel and host compute the layout from this)
__host__ __device__ constexpr uint32_t exact_fixed_smem(uint32_t k_chunks, bool stream_a) {
  return (stream_a ? 0u : k_chunks * kChunkBytes) + kEpiWarps * kWq * 12 + 32 * 8 + 16;
}

struct ExactArgs {
  uint32_t n_vec, nq, k_chunks;
  uint32_t n_stages;              // B pipeline stages (2..kMaxStages)
  uint32_t fp16;                  // operand format: 1 FP16, 0 BF16 (instruction descriptor a_format / b_format)
  uint32_t stream_a;              // 1: A (the query block) is not resident; its K chunk travels in every stage, ahead
                                  //    of the B chunk (dims above 512: 128 x K BF16 no longer fits beside the pipeline)
  uint32_t tile_lo, tile_hi;      // vector tiles of this pass
  uint32_t tiles_per_item;        // consecutive tiles one CTA (pair) handles for one query block
  uint32_t n_qblocks, n_items;    // query blocks: 128 queries each, 256 (two CTAs x 128) in the two-CTA form
  const float* thresh;            // [nq] keep keys >= thresh
  uint32_t* cand_cnt;             // [nq]
  uint32_t* cand_id;              // [nq][cap]
  float* cand_key;                // [nq][cap]
  uint32_t cap;
  uint32_t* qflags;               // [nq] bit 0: this query lost a candidate (buffer full) -> redone by the streaming scan
  unsigned long long* dbg;  // optional [16] cycle counters (diagnostics)
  uint32_t dense;           // first slice (every threshold is -inf): each key goes straight to its column's slot of the
                            // query's buffer (position = column - first column of the slice); the host presets cand_cnt
  uint32_t diag;            // measurement only (TURDB_EXACT_DIAG; results are WRONG when set): 1 = the epilogue never reads
                            // TMEM, 2 = it reads the accumulator but looks at nothing
};

// ---- two-CTA (cta_group::2) helpers ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {  // same offset in CTA `rank` of the cluster
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load whose completion is counted on a barrier of EITHER CTA of the pair (`bar` is a shared::cluster address)
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, int32_t c0, int32_t c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tc_commit_pair(uint32_t bar) {  // arrives on `bar`'s offset in BOTH CTAs of the pair
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ void tc_mma_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Remote arrive on the leader's "accumulator drained" barrier.  No generic-memory data travels through it — what it
// orders is this warp's TMEM reads (complete after tcgen05.wait::ld, fenced by tcgen05.fence::before_thread_sync) against
// the tensor pipe's next writes — so the default CTA-scope form is enough; the .release.cluster form (a cluster-wide
// fence per arrive) was the most-sampled line of the two-CTA kernel (38 % of all samples, ncu).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ bool elect_one() {  // true in exactly one lane of the (converged) warp
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ float max8(const uint32_t* v) {
  const float a = fmaxf(fmaxf(__uint_as_float(v[0]), __uint_as_float(v[1])), __uint_as_float(v[2]));
  const float b = fmaxf(fmaxf(__uint_as_float(v[3]), __uint_as_float(v[4])), __uint_as_float(v[5]));
  return fmaxf(fmaxf(a, b), fmaxf(__uint_as_float(v[6]), __uint_as_float(v[7])));
}

// Flush of a warp's candidate queue (rare path, kept out of line): entry i belongs to query q_base + q_lane[i]; lane i
// reserves a slot in that query's buffer with its own atomicAdd, so up to 64 candidates cost one round trip.
__device__ __noinline__ void exact_wq_flush(uint32_t* cand_cnt, uint32_t* cand_id, float* cand_key, uint32_t* qflags, uint32_t cap,
                                            const float* q_key, const uint32_t* q_id, const uint32_t* q_lane, uint32_t q_base,
                                            uint32_t n) {
  const uint32_t lane = threadIdx.x & 31;
  __syncwarp();
  for (uint32_t i = lane; i < n; i += 32) {
    const uint32_t q = q_base + q_lane[i];
    const uint32_t pos = atomicAdd(cand_cnt + q, 1u);
    if (pos < cap) {
      cand_id[(size_t)q * cap + pos] = q_id[i];
      cand_key[(size_t)q * cap + pos] = q_key[i];
    } else {
      qflags[q] = 1u;
    }
  }
  __syncwarp();
}

// smem: [A: k_chunks x 16 KB (resident form)][stages: n_stages x ([A chunk] B chunk)]
//       [warp queues: key | id | lane][barriers][tmem ptr]
template <bool STREAM_A, bool PAIR, uint32_t TILE_N>
__device__ __forceinline__ void exact_gemm_filter_body(const CUtensorMap* map_q, const CUtensorMap* map_x, const ExactArgs& a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;   // CTA within the pair; rank 0 (the leader) issues the MMAs
  const uint32_t n_workers = PAIR ? gridDim.x >> 1 : gridDim.x, worker = PAIR ? blockIdx.x >> 1 : blockIdx.x;
  // TILE_N = 256 (shipped): two 256-column accumulators, every epilogue warp on every tile.  TILE_N = 128 (measured
  // alternative, TURDB_EXACT_TILE_N=128): FOUR 128-column accumulators and two alternating sets of eight epilogue warps (set
  // s takes the tiles with sequence number = s mod 2), so that every accumulator hand-off (commit -> wake -> TMEM load ->
  // arrive -> wake, ~0.9k cycles against ~1k cycles of MMAs per 256-column tile at K = 128) has three tiles of cover.
  // Parity-green and slower at every short K tried (128-d L2 4.63 against 3.26 ms): twice the MMA instructions, commits and
  // barrier round trips per score.
  constexpr uint32_t kBufs = 512 / TILE_N;                          // accumulator buffers in TMEM
  constexpr uint32_t kSets = TILE_N == 128 ? 2 : 1;                 // alternating sets of epilogue warps
  static_assert(TILE_N == 128 || TILE_N == 256, "UMMA N");
  static_assert((kEpiWarps / kSets) * kEpiCols == 4 * TILE_N, "a set's warps cover the tile: 4 lane quarters x TILE_N columns");
  constexpr uint32_t kBRows = PAIR ? TILE_N / 2 : TILE_N;          // vector rows this CTA stages per tile
  constexpr uint32_t stage_bytes = exact_stage_bytes(STREAM_A, PAIR, TILE_N);  // [A chunk |] B chunk
  constexpr uint32_t b_in_stage = STREAM_A ? kChunkBytes : 0;
  constexpr uint32_t kQRows = PAIR ? 2 * kTileM : kTileM;          // queries per work item
  uint8_t* sA = smem;
  uint8_t* sB = sA + (STREAM_A ? 0 : (size_t)a.k_chunks * kChunkBytes);
  const uint32_t kStages = a.n_stages;
  float* wq_key = reinterpret_cast<float*>(sB + (size_t)kStages * stage_bytes);  // [kEpiWarps][kWq]
  uint32_t* wq_id = reinterpret_cast<uint32_t*>(wq_key + kEpiWarps * kWq);
  uint32_t* wq_lane = wq_id + kEpiWarps * kWq;
  uint64_t* bars = reinterpret_cast<uint64_t*>(wq_lane + kEpiWarps * kWq);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 32);
  const uint32_t bar_a_full = smem_u32(bars + 0), bar_a_empty = smem_u32(bars + 1);
  const uint32_t bar_b_full = smem_u32(bars + 2), bar_b_empty = smem_u32(bars + 2 + kMaxStages);
  const uint32_t bar_t_full = smem_u32(bars + 2 + 2 * kMaxStages), bar_t_empty = smem_u32(bars + 6 + 2 * kMaxStages);  // 4 + 4 slots

  if (threadIdx.x == 0) {
    mbar_init(bar_a_full, 1);
    mbar_init(bar_a_empty, 1);
    for (uint32_t s = 0; s < kStages; ++s) {
      mbar_init(bar_b_full + 8 * s, 1);
      mbar_init(bar_b_empty + 8 * s, 1);
    }
    for (uint32_t s = 0; s < kBufs; ++s) {
      mbar_init(bar_t_full + 8 * s, 1);
      mbar_init(bar_t_empty + 8 * s, (PAIR ? 2 : 1) * (kEpiWarps / kSets));  // one arrive per warp of the tile's set (of both CTAs)
    }
    mbar_fence_init();
  }
  if (warp == 1) {  // kBufs accumulator buffers x TILE_N FP32 columns = all 512 (in each CTA of a pair)
    if (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  if (PAIR) cluster_sync_all();  // the peer's barriers exist before anything signals them
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const unsigned long long k_t0 = a.dbg ? (unsigned long long)clock64() : 0ull;

  // The two single-issuer roles run with the WHOLE warp converged (every lane evaluates the loop control and the waits,
  // one elected lane issues): all addresses and descriptors are then warp-uniform, so the compiler keeps them in uniform
  // registers — inside an `if (lane == 0)` region it had to broadcast every operand of every tcgen05.mma through an
  // ELECT / R2UR / BRA.U.ANY loop (~16 instructions per MMA), which at K = 128 (8 MMAs per tile) made the issuer thread
  // itself the pace of the tensor pipe.
  if (warp == 0) {
    // ===== TMA producer (in BOTH CTAs of a pair: own queries, own half of the vector tile) =====
    {
      // completions are counted on the leader's barriers; only the leader arms them (with both CTAs' bytes)
      const uint32_t full_a = PAIR ? mapa_u32(bar_a_full, 0) : bar_a_full;
      const uint32_t full_b = PAIR ? mapa_u32(bar_b_full, 0) : bar_b_full;
      const uint32_t n_arm = PAIR ? 2u : 1u;
      uint32_t stage = 0, phase = 0, a_phase = 0;
      for (uint32_t item = worker; item < a.n_items; item += n_workers) {
        const uint32_t qb = item % a.n_qblocks;
        const int32_t q_row0 = (int32_t)(qb * kQRows + rank * kTileM);
        const uint32_t t0 = a.tile_lo + (item / a.n_qblocks) * a.tiles_per_item;
        const uint32_t t1 = min(a.tile_hi, t0 + a.tiles_per_item);
        if (!STREAM_A) {
          long long c0 = a.dbg ? clock64() : 0;
          mbar_wait(bar_a_empty, a_phase ^ 1);  // previous item's MMAs have drained A
          if (a.dbg && lane == 0) atomicAdd(a.dbg + 0, (unsigned long long)(clock64() - c0));
          if (elect_one()) {
            if (rank == 0) mbar_expect_tx(bar_a_full, n_arm * a.k_chunks * kChunkBytes);
            for (uint32_t kc = 0; kc < a.k_chunks; ++kc) {
              if (PAIR) tma_load_2d_pair(smem_u32(sA + (size_t)kc * kChunkBytes), map_q, (int32_t)(kc * kChunkK), q_row0, full_a);
              else tma_load_2d(smem_u32(sA + (size_t)kc * kChunkBytes), map_q, (int32_t)(kc * kChunkK), q_row0, full_a);
            }
          }
          __syncwarp();
          a_phase ^= 1;
        }
        for (uint32_t t = t0; t < t1; ++t) {
          const int32_t x_row0 = (int32_t)(t * TILE_N + rank * kBRows);
          for (uint32_t kc = 0; kc < a.k_chunks; ++kc) {
            long long c1 = a.dbg ? clock64() : 0;
            mbar_wait(bar_b_empty + 8 * stage, phase ^ 1);
            if (a.dbg && lane == 0) atomicAdd(a.dbg + 1, (unsigned long long)(clock64() - c1));
            if (elect_one()) {
              if (rank == 0) mbar_expect_tx(bar_b_full + 8 * stage, n_arm * stage_bytes);
              const uint32_t dst = smem_u32(sB + (size_t)stage * stage_bytes);
              if (PAIR) {
                if (STREAM_A) tma_load_2d_pair(dst, map_q, (int32_t)(kc * kChunkK), q_row0, full_b + 8 * stage);
                tma_load_2d_pair(dst + b_in_stage, map_x, (int32_t)(kc * kChunkK), x_row0, full_b + 8 * stage);
              } else {
                if (STREAM_A)  // the query block's chunk comes from L2 (it is 128 x K, re-read once per vector tile)
                  tma_load_2d(dst, map_q, (int32_t)(kc * kChunkK), q_row0, full_b + 8 * stage);
                tma_load_2d(dst + b_in_stage, map_x, (int32_t)(kc * kChunkK), x_row0, full_b + 8 * stage);
              }
            }
            __syncwarp();
            if (++stage == kStages) {
              stage = 0;
              phase ^= 1;
            }
          }
        }
      }
      // drain: every stage (and A) has been released, i.e. every commit aimed at this CTA's barriers has landed —
      // a CTA of a pair must not exit while its peer's tensor pipe can still signal it
      for (uint32_t s = 0; s < kStages; ++s) {
        mbar_wait(bar_b_empty + 8 * stage, phase ^ 1);
        if (++stage == kStages) {
          stage = 0;
          phase ^= 1;
        }
      }
      if (!STREAM_A) mbar_wait(bar_a_empty, a_phase ^ 1);
    }
  } else if (warp == 1) {
    // ===== MMA issuer (one elected lane; in a pair only the leader CTA's) =====
    if (rank == 0) {
      // instruction descriptor: D=F32, A=B=F16/BF16, both K-major, N, M (cute::UMMA::InstrDescriptor); M = 256 across a pair
      const uint32_t fmt = a.fp16 ? 0u : 1u;  // a_format (bits 7-9) / b_format (bits 10-12): 0 = F16, 1 = BF16
      const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((TILE_N >> 3) << 17) | (((PAIR ? 2 * kTileM : kTileM) >> 4) << 24);
      uint32_t stage = 0, phase = 0, a_phase = 0, acc = 0, acc_phase = 0;
      for (uint32_t item = worker; item < a.n_items; item += n_workers) {
        const uint32_t t0 = a.tile_lo + (item / a.n_qblocks) * a.tiles_per_item;
        const uint32_t t1 = min(a.tile_hi, t0 + a.tiles_per_item);
        if (!STREAM_A) {
          long long c2 = a.dbg ? clock64() : 0;
          mbar_wait(bar_a_full, a_phase);
          if (a.dbg && lane == 0) atomicAdd(a.dbg + 2, (unsigned long long)(clock64() - c2));
          a_phase ^= 1;
        }
        tc_fence_after();
        for (uint32_t t = t0; t < t1; ++t) {
          long long c3 = a.dbg ? clock64() : 0;
          mbar_wait(bar_t_empty + 8 * acc, acc_phase ^ 1);  // the epilogue (of both CTAs of a pair) has drained this accumulator
          if (a.dbg && lane == 0) atomicAdd(a.dbg + 3, (unsigned long long)(clock64() - c3));
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + acc * TILE_N;
          for (uint32_t kc = 0; kc < a.k_chunks; ++kc) {
            long long c4 = a.dbg ? clock64() : 0;
            mbar_wait(bar_b_full + 8 * stage, phase);
            if (a.dbg && lane == 0) atomicAdd(a.dbg + 4, (unsigned long long)(clock64() - c4));
            tc_fence_after();
            const uint64_t da = umma_desc_sw128(STREAM_A ? smem_u32(sB + (size_t)stage * stage_bytes)
                                                           : smem_u32(sA + (size_t)kc * kChunkBytes));
            const uint64_t db = umma_desc_sw128(smem_u32(sB + (size_t)stage * stage_bytes + b_in_stage));
            if (elect_one()) {
#pragma unroll
              for (uint32_t k4 = 0; k4 < kChunkK / 16; ++k4) {  // UMMA_K = 16 elements = 32 B inside the swizzle row
                if (PAIR) tc_mma_pair(d_tmem, da + 2 * k4, db + 2 * k4, idesc, (kc | k4) != 0 ? 1u : 0u);
                else tc_mma_bf16(d_tmem, da + 2 * k4, db + 2 * k4, idesc, (kc | k4) != 0 ? 1u : 0u);
              }
              if (PAIR) tc_commit_pair(bar_b_empty + 8 * stage);  // frees the stage (in both CTAs) when these MMAs retire
              else tc_commit(bar_b_empty + 8 * stage);
            }
            __syncwarp();
            if (++stage == kStages) {
              stage = 0;
              phase ^= 1;
            }
          }
          if (elect_one()) {
            if (PAIR) tc_commit_pair(bar_t_full + 8 * acc);
            else tc_commit(bar_t_full + 8 * acc);
            if (a.dbg) atomicAdd(a.dbg + 5, 1ull);  // tiles
          }
          __syncwarp();
          if (++acc == kBufs) {
            acc = 0;
            acc_phase ^= 1;
          }
        }
        if (!STREAM_A) {
          if (elect_one()) {
            if (PAIR) tc_commit_pair(bar_a_empty);
            else tc_commit(bar_a_empty);
          }
          __syncwarp();
        }
      }
    }
  } else {
    // ===== epilogue: kEpiWarps warps; warp = one TMEM lane quarter (32 query rows) x kEpiCols of the tile's columns =====
    // (Measured and dropped: two alternating SETS of eight warps, set s serving accumulator s with two rounds of kEpiCols
    // per tile — the same work in another order: 128-d 3.32 against 3.19 ms, 768-d 10.36 against 10.20 ms.  At short K the
    // tensor pipe idles on the accumulator hand-offs — commit -> wake -> TMEM load -> arrive -> wake, ~0.9k cycles per
    // 1.05k-cycle tile at 128-d (ncu: pipe 53 % active, the issuer 29 % of its time on bar_t_empty) — which two
    // 256-column buffers cannot hide.  Four 128-column buffers (TILE_N = 128 below) hide them and still lose: 4.63 against
    // 3.26 ms at 128-d L2.)
    const uint32_t ew = warp - 2;                    // index among the epilogue warps
    const uint32_t quarter = warp & 3;               // TMEM lane quarter this warp may read (= warp id % 4)
    const uint32_t set = kSets == 2 ? ew / (kEpiWarps / 2) : 0u;              // which tiles this warp takes (sequence % kSets)
    const uint32_t cslice = ((ew % (kEpiWarps / kSets)) >> 2) * kEpiCols;     // first tile column of this warp's slice
    const uint32_t et = threadIdx.x - 64;            // index among the epilogue threads
    const uint32_t lt_mask = (1u << lane) - 1u;
    float* my_key = wq_key + ew * kWq;
    uint32_t* my_id = wq_id + ew * kWq;
    uint32_t* my_lane = wq_lane + ew * kWq;
    const uint32_t t_empty_dst = PAIR ? mapa_u32(bar_t_empty, 0) : bar_t_empty;  // the leader's barrier
    uint32_t seq = 0;                                // tiles this CTA has started, all items: tile seq uses buffer seq % kBufs
    uint32_t wq_n = 0;                               // entries in the warp's queue (warp-uniform)
    uint32_t q_base = 0;                             // query of queue entry i = q_base + my_lane[i]
    auto flush = [&]() {                             // whole warp: entry i is written out by lane i (and i + 32)
      exact_wq_flush(a.cand_cnt, a.cand_id, a.cand_key, a.qflags, a.cap, my_key, my_id, my_lane, q_base, wq_n);
      wq_n = 0;
    };
    for (uint32_t item = worker; item < a.n_items; item += n_workers) {
      const uint32_t qb = item % a.n_qblocks;
      const uint32_t t0 = a.tile_lo + (item / a.n_qblocks) * a.tiles_per_item;
      const uint32_t t1 = min(a.tile_hi, t0 + a.tiles_per_item);
      q_base = qb * kQRows + rank * kTileM + quarter * 32;
      const uint32_t q = q_base + lane;
      const float tau = q < a.nq ? a.thresh[q] : INFINITY;  // rows past the batch never keep anything
      for (uint32_t t = t0; t < t1; ++t, ++seq) {
        if (kSets == 2 && (seq & 1u) != set) continue;  // the other set's tile
        const uint32_t acc = seq % kBufs, acc_phase = (seq / kBufs) & 1u;
        long long c6 = (a.dbg && et == 0) ? clock64() : 0;
        mbar_wait(bar_t_full + 8 * acc, acc_phase);
        long long c7 = (a.dbg && et == 0) ? clock64() : 0;
        tc_fence_after();
        const uint32_t n_valid = min(TILE_N, a.n_vec - t * TILE_N);  // columns past the corpus are zero rows
        uint32_t v[kEpiCols / 32][32];
        const uint32_t tcol = tmem_base + ((quarter * 32) << 16) + acc * TILE_N + cslice;
        if (a.diag != 1) {
#pragma unroll
          for (uint32_t cb = 0; cb < kEpiCols / 32; ++cb) tmem_ld_32x32b_x32_nowait(tcol + cb * 32, v[cb]);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        } else {
#pragma unroll
          for (uint32_t cb = 0; cb < kEpiCols / 32; ++cb)
#pragma unroll
            for (uint32_t j = 0; j < 32; ++j) v[cb][j] = 0xff800000u;  // -inf: nothing passes
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {  // the tensor pipe may refill this accumulator now
          if (PAIR) mbar_arrive_cluster(t_empty_dst + 8 * acc);
          else mbar_arrive(t_empty_dst + 8 * acc);
        }
        if (a.diag == 2) continue;
#pragma unroll
        for (uint32_t cb = 0; cb < kEpiCols / 32; ++cb) {
          if (a.dense) {  // first slice: no test, no queue — 128-bit stores of the thread's 32 consecutive columns
            if (q < a.nq) {
              const uint32_t c0 = cslice + cb * 32;  // tile column of v[cb][0]
              const size_t slot = (size_t)q * a.cap + (size_t)(t - a.tile_lo) * TILE_N + c0;
              float4* kd = reinterpret_cast<float4*>(a.cand_key + slot);
              uint4* idd = reinterpret_cast<uint4*>(a.cand_id + slot);
#pragma unroll
              for (uint32_t j = 0; j < 32; j += 4) {
                float4 kv;
                kv.x = __uint_as_float(v[cb][j]);
                kv.y = __uint_as_float(v[cb][j + 1]);
                kv.z = __uint_as_float(v[cb][j + 2]);
                kv.w = __uint_as_float(v[cb][j + 3]);
                // a NaN score (0 x inf against an absent vector's +inf marker) must not win the selection
                kv.x = kv.x == kv.x ? kv.x : -INFINITY;
                kv.y = kv.y == kv.y ? kv.y : -INFINITY;
                kv.z = kv.z == kv.z ? kv.z : -INFINITY;
                kv.w = kv.w == kv.w ? kv.w : -INFINITY;
                kd[j >> 2] = kv;
                const uint32_t id0 = t * TILE_N + c0 + j;
                idd[j >> 2] = make_uint4(id0, id0 + 1, id0 + 2, id0 + 3);
              }
            }
            continue;
          }
          // a key that reaches the running threshold is rare once the first slices have been seen
          float g[4];
#pragma unroll
          for (uint32_t gi = 0; gi < 4; ++gi) g[gi] = max8(&v[cb][8 * gi]);
          const float m = fmaxf(fmaxf(g[0], g[1]), fmaxf(g[2], g[3]));
          if (__any_sync(kFullMask, m >= tau)) {
#pragma unroll
            for (uint32_t gi = 0; gi < 4; ++gi) {
              if (__any_sync(kFullMask, g[gi] >= tau)) {
#pragma unroll
                for (uint32_t j = 0; j < 8; ++j) {
                  const uint32_t col = cslice + cb * 32 + gi * 8 + j;  // tile column
                  const float key = __uint_as_float(v[cb][gi * 8 + j]);
                  const bool hit = key >= tau && col < n_valid;
                  const uint32_t b = __ballot_sync(kFullMask, hit);
                  if (b) {
                    if (hit) {
                      const uint32_t slot = wq_n + __popc(b & lt_mask);
                      my_key[slot] = key;
                      my_id[slot] = t * TILE_N + col;
                      my_lane[slot] = lane;
                    }
                    wq_n += __popc(b);
                    if (wq_n > 32) flush();
                  }
                }
              }
            }
          }
        }
        if (a.dbg && et == 0) {
          atomicAdd(a.dbg + 6, (unsigned long long)(c7 - c6));
          atomicAdd(a.dbg + 7, (unsigned long long)(clock64() - c7));
        }
      }
      if (wq_n) flush();  // the queue's entries are relative to this item's query block
    }
  }

  if (a.dbg && threadIdx.x == 0) atomicAdd(a.dbg + 8, (unsigned long long)clock64() - k_t0);
  tc_fence_before();
  __syncwarp();
  if (PAIR) cluster_sync_all();  // neither CTA leaves (or frees TMEM) while the other can still touch it
  else __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    if (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

template <bool STREAM_A, uint32_t TILE_N>
__global__ void __launch_bounds__(kExactThreads, 1)
exact_gemm_filter_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_x,
                         const ExactArgs a) {
  exact_gemm_filter_body<STREAM_A, false, TILE_N>(&map_q, &map_x, a);
}

// the two-CTA form: clusters of 2 CTAs (one TPC), grid = 2 x the number of pairs
template <bool STREAM_A, uint32_t TILE_N>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kExactThreads, 1)
exact_gemm_filter_pair_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_x,
                              const ExactArgs a) {
  exact_gemm_filter_body<STREAM_A, true, TILE_N>(&map_q, &map_x, a);
}

// ------------------------------------------------------------------------------------------------
// pass (2): per query, new threshold = (kprime-th best filter key so far) - slack; keep every key above it
// ------------------------------------------------------------------------------------------------
// One WARP per query, no block barriers.  The buffer holds [0, kept[q]) = what the previous call kept, then this slice's
// arrivals.  The kprime-th best key is found by a 4-digit radix select over the order-preserving integer image of the
// keys (one 256-bin histogram per warp in shared memory, votes aggregated with match.any so that keys sharing an
// exponent byte cost one atomic); everything at or above tau' = that key - 2 e(q) is compacted to the front of the
// buffer in place (stable: a ballot per 32 entries).  (The first version sorted the whole buffer with a bitonic network in
// shared memory, 45 block barriers for 512 entries: 0.13-0.55 ms per pass for 10k queries; nothing downstream needs
// the order — the rerank sorts by FP32 distance, the SQL operator replays the archive.)
// With `arch_id` the arrivals are first appended to the query's archive (ids only, never pruned): the union of all
// arrivals is a superset of the rows a sequential scan would ever have pushed into its top-K heap (sql_topk.inl replays
// exactly that).  A query whose buffer or archive overflowed is flagged (qflags[q]) and redone by the streaming scan.
__device__ __forceinline__ uint32_t key_to_ordered(float f) {  // larger key <=> larger integer
  const uint32_t b = __float_as_uint(f);
  return b ^ ((b >> 31) ? 0xFFFFFFFFu : 0x80000000u);
}
__device__ __forceinline__ float ordered_to_key(uint32_t u) {
  return __uint_as_float((u & 0x80000000u) ? (u ^ 0x80000000u) : ~u);
}
constexpr uint32_t kThreshWarps = 4;
__global__ void __launch_bounds__(32 * kThreshWarps) exact_threshold_kernel(uint32_t nq, uint32_t kprime, uint32_t cap,
                                                                            uint32_t* cand_cnt, uint32_t* cand_id, float* cand_key,
                                                                            float* thresh, const float* __restrict__ slack,
                                                                            uint32_t* kept, uint32_t* qflags, uint32_t* arch_cnt,
                                                                            uint32_t* arch_id, uint32_t arch_cap,
                                                                            const uint64_t* __restrict__ live) {
  __shared__ uint32_t hist[kThreshWarps][256];
  const uint32_t w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t q = blockIdx.x * kThreshWarps + w;
  if (q >= nq) return;  // whole warps leave; nothing below synchronises across warps
  uint32_t* h = hist[w];
  const uint32_t lt_mask = (1u << lane) - 1u;
  const uint32_t raw_cnt = cand_cnt[q];
  const uint32_t cnt = min(raw_cnt, cap);
  const uint32_t prev = min(kept[q], cnt);
  bool flag = raw_cnt > cap;
  float* keys = cand_key + (size_t)q * cap;
  uint32_t* ids = cand_id + (size_t)q * cap;
  // deleted rows (live bit clear; live == null: none) are dropped here, so nothing downstream sees them: they are
  // neither archived nor kept, and tau is the kprime-th best LIVE key
  auto is_live = [&](uint32_t id) { return !live || ((live[id >> 6] >> (id & 63)) & 1ull) != 0; };
  if (arch_id) {
    const uint32_t base = arch_cnt[q];
    uint32_t n_new = 0;
    for (uint32_t b = prev; b < cnt; b += 32) {
      const uint32_t i = b + lane;
      const uint32_t id = i < cnt ? ids[i] : 0u;
      const bool ok = i < cnt && is_live(id);
      const uint32_t bal = __ballot_sync(kFullMask, ok);
      const uint32_t pos = base + n_new + __popc(bal & lt_mask);
      if (ok && pos < arch_cap) arch_id[(size_t)q * arch_cap + pos] = id;
      n_new += __popc(bal);
    }
    __syncwarp();
    if (lane == 0) arch_cnt[q] = min(base + n_new, arch_cap);
    if (base + n_new > arch_cap) flag = true;
  }
  uint32_t n_live = cnt;
  if (live) {
    n_live = 0;
    for (uint32_t b = 0; b < cnt; b += 32) n_live += __popc(__ballot_sync(kFullMask, b + lane < cnt && is_live(ids[b + lane])));
  }
  float tau = -INFINITY;
  if (kprime > 0 && n_live >= kprime) {
    uint32_t prefix = 0, remaining = kprime;  // the remaining-th largest among the keys whose high digits equal prefix
    for (int shift = 24; shift >= 0; shift -= 8) {
      for (uint32_t i = lane; i < 256; i += 32) h[i] = 0;
      __syncwarp();
      const uint32_t hi_mask = shift == 24 ? 0u : (0xFFFFFFFFu << (shift + 8));
      for (uint32_t base = 0; base < cnt; base += 32) {
        const uint32_t i = base + lane;
        bool ok = i < cnt;
        uint32_t u = 0;
        if (ok) {
          u = key_to_ordered(keys[i]);
          ok = (u & hi_mask) == prefix && is_live(ids[i]);
        }
        const uint32_t digit = (u >> shift) & 255u;
        const uint32_t active = __ballot_sync(kFullMask, ok);
        if (ok) {
          const uint32_t peers = __match_any_sync(active, digit);
          if ((uint32_t)(__ffs(peers) - 1) == lane) atomicAdd(&h[digit], (uint32_t)__popc(peers));
        }
      }
      __syncwarp();
      // lane l owns the 8 bins 255 - 8l ... 248 - 8l (lane 0 = the largest digits); prefix sums run from the top
      uint32_t b[8], mine = 0;
#pragma unroll
      for (uint32_t j = 0; j < 8; ++j) {
        b[j] = h[255 - (8 * lane + j)];
        mine += b[j];
      }
      uint32_t incl = mine;
#pragma unroll
      for (uint32_t off = 1; off < 32; off <<= 1) {
        const uint32_t t = __shfl_up_sync(kFullMask, incl, off);
        if (lane >= off) incl += t;
      }
      const uint32_t excl = incl - mine;
      const bool here = excl < remaining && remaining <= incl;  // exactly one lane (the matching keys number >= remaining)
      uint32_t f_digit = 0, f_rem = 0, c = excl;
      bool done = false;
#pragma unroll
      for (uint32_t j = 0; j < 8; ++j) {
        if (here && !done && c + b[j] >= remaining) {
          f_digit = 255 - (8 * lane + j);
          f_rem = remaining - c;
          done = true;
        }
        c += b[j];
      }
      const uint32_t src = (uint32_t)__ffs(__ballot_sync(kFullMask, here)) - 1u;
      f_digit = __shfl_sync(kFullMask, f_digit, src & 31u);
      remaining = __shfl_sync(kFullMask, f_rem, src & 31u);
      prefix |= f_digit << shift;
      __syncwarp();
    }
    // tau' = kprime-th best key - 2 e(q); everything at or above it stays (>= kprime entries)
    tau = ordered_to_key(prefix) - (slack ? slack[q] : 0.f);
  }
  uint32_t keep = 0;
  for (uint32_t base = 0; base < cnt; base += 32) {
    const uint32_t i = base + lane;
    float kf = 0.f;
    uint32_t id = 0;
    bool ok = false;
    if (i < cnt) {
      kf = keys[i];
      id = ids[i];
      ok = kf >= tau && is_live(id);
    }
    const uint32_t bal = __ballot_sync(kFullMask, ok);
    __syncwarp();  // every lane has read its entry before any lane overwrites one (targets are <= own index)
    if (ok) {
      const uint32_t pos = keep + __popc(bal & lt_mask);
      if (pos < cap / 2) {
        keys[pos] = kf;
        ids[pos] = id;
      }
    }
    keep += __popc(bal);
    __syncwarp();
  }
  if (keep > cap / 2) {  // no room left for the next slice's arrivals: give the query to the streaming scan
    keep = cap / 2;
    flag = true;
  }
  if (lane == 0) {
    cand_cnt[q] = keep;
    kept[q] = keep;
    thresh[q] = tau;
    if (flag) qflags[q] = 1u;
  }
}

// ------------------------------------------------------------------------------------------------
// pass (3): FP32 rerank in the reference's lane order + final ascending top-k
// ------------------------------------------------------------------------------------------------
// One CTA (128 threads = 32 quads) per query.  Distances follow select_squared_distance_fn; ties order by node id.
template <int METRIC>
__global__ void __launch_bounds__(128) exact_rerank_kernel(DeviceIndex ix, const float* __restrict__ queries, uint32_t nq,
                                                           uint32_t k, uint32_t cap, const uint32_t* __restrict__ cand_cnt,
                                                           const uint32_t* __restrict__ cand_id,
                                                           const uint32_t* __restrict__ qflags, uint64_t* out_rows,
                                                           uint32_t* out_nodes, float* out_dist, uint32_t* out_counts) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const uint32_t q = blockIdx.x;
  if (q >= nq) return;
  if (qflags[q]) return;  // a candidate was lost (buffer full): exact_stream_topk_kernel redoes this query
  const uint32_t cnt = min(cand_cnt[q], cap);
  uint32_t n2 = 1;
  while (n2 < cnt) n2 <<= 1;
  float* qs = reinterpret_cast<float*>(smem_raw);           // [ds]
  float* sd = qs + ix.ds;                                   // [n2]
  uint32_t* si = reinterpret_cast<uint32_t*>(sd + n2);      // [n2]
  for (uint32_t i = threadIdx.x; i < ix.ds; i += blockDim.x) qs[i] = i < ix.dim ? queries[(size_t)q * ix.dim + i] : 0.f;
  __syncthreads();
  const uint32_t p = threadIdx.x & 3, quad = threadIdx.x >> 2;
  const float qn = (METRIC == kCosine) ? quad_dot(qs, qs, ix.dim, p) : 0.f;
  for (uint32_t base = 0; base < n2; base += 32) {
    const uint32_t c = base + quad;
    const uint32_t id = c < cnt ? cand_id[(size_t)q * cap + c] : 0u;
    const float* b = ix.arena + (size_t)id * ix.ds;
    float raw = (METRIC == kL2) ? quad_l2sq(qs, b, ix.dim, p) : quad_dot(qs, b, ix.dim, p);
    if (p == 0 && c < n2) {
      float d = raw;
      if (METRIC == kIP) d = -raw;
      if (METRIC == kCosine) d = cosine_finish(raw, qn, ix.norm2[id]);
      if (b[0] == INFINITY) d = INFINITY;  // absent vector
      sd[c] = c < cnt ? d : INFINITY;
      si[c] = c < cnt ? id : 0xFFFFFFFFu;
    }
  }
  __syncthreads();
  for (uint32_t size = 2; size <= n2; size <<= 1) {
    for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
      for (uint32_t i = threadIdx.x; i < n2; i += blockDim.x) {
        const uint32_t j = i ^ stride;
        if (j > i) {
          const bool asc = (i & size) == 0;
          const float di = sd[i], dj = sd[j];
          const uint32_t ii = si[i], ij = si[j];
          const bool i_first = di < dj || (di == dj && ii < ij);
          if (i_first != asc) {
            sd[i] = dj; sd[j] = di;
            si[i] = ij; si[j] = ii;
          }
        }
      }
      __syncthreads();
    }
  }
  const uint32_t count = min(cnt, k);
  for (uint32_t i = threadIdx.x; i < k; i += blockDim.x) {
    const size_t o = (size_t)q * k + i;
    if (i < count) {
      out_rows[o] = ix.row_ids[si[i]];
      if (out_nodes) out_nodes[o] = si[i];
      out_dist[o] = sd[i];
    } else {
      out_rows[o] = 0xFFFFFFFFFFFFFFFFull;
      if (out_nodes) out_nodes[o] = kInvalid;
      out_dist[o] = INFINITY;
    }
  }
  if (threadIdx.x == 0) out_counts[q] = count;
}

// The scan itself, for the queries the filter could not serve (qflags[q] != 0): FP32 distances in the reference's lane
// order over ALL rows, top-k by (distance, node id).  CTAs stride over the queries and skip unflagged ones; always
// enqueued, exits at once when nothing is flagged.  smem: query [ds] | list d [k] | list id [k] | chunk d [64]
template <int METRIC>
__global__ void __launch_bounds__(256) exact_stream_topk_kernel(DeviceIndex ix, const float* __restrict__ queries, uint32_t nq,
                                                                uint32_t k, const uint32_t* __restrict__ qflags,
                                                                uint64_t* out_rows, uint32_t* out_nodes, float* out_dist,
                                                                uint32_t* out_counts) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  float* qs = reinterpret_cast<float*>(smem_raw);
  float* ld = qs + ix.ds;
  uint32_t* li = reinterpret_cast<uint32_t*>(ld + k);
  float* cd = reinterpret_cast<float*>(li + k);
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, p = tid & 3, quad = tid >> 2;
  for (uint32_t q = blockIdx.x; q < nq; q += gridDim.x) {
    if (!qflags[q]) continue;
    __syncthreads();
    for (uint32_t i = tid; i < ix.ds; i += blockDim.x) qs[i] = i < ix.dim ? queries[(size_t)q * ix.dim + i] : 0.f;
    __syncthreads();
    const float qn = (METRIC == kCosine) ? quad_dot(qs, qs, ix.dim, p) : 0.f;
    uint32_t len = 0;  // meaningful in warp 0
    for (uint64_t base = 0; base < ix.n; base += 64) {
      const uint64_t r = min(base + quad, ix.n - 1);
      const float* b = ix.arena + r * ix.ds;
      const float raw = (METRIC == kL2) ? quad_l2sq(qs, b, ix.dim, p) : quad_dot(qs, b, ix.dim, p);
      if (p == 0) {
        float d = raw;
        if (METRIC == kIP) d = -raw;
        if (METRIC == kCosine) d = cosine_finish(raw, qn, ix.norm2[r]);
        if (b[0] == INFINITY) d = INFINITY;
        cd[quad] = d;
      }
      __syncthreads();
      if (warp == 0) {
        const uint32_t cnt = (uint32_t)min((uint64_t)64, (uint64_t)(ix.n - base));
        const uint64_t lw = ix.live ? ix.live[base >> 6] : ~0ull;  // the chunk is one word of the live bitmap
        for (uint32_t half = 0; half < cnt; half += 32) {
          const uint32_t j = half + lane;
          const float dj = j < cnt ? cd[j] : INFINITY;
          uint32_t mask = __ballot_sync(kFullMask, j < cnt && ((lw >> j) & 1ull) && (len < k || dj < ld[k - 1]));
          while (mask) {
            const uint32_t l = __ffs(mask) - 1;
            mask &= mask - 1;
            const float d = cd[half + l];
            const uint32_t id = (uint32_t)(base + half + l);
            if (len < k || d < ld[len - 1]) {
              // position = entries with distance <= d (they hold smaller node ids: rows arrive in ascending order)
              uint32_t c = 0;
              for (uint32_t i = lane; i < len; i += 32) c += (ld[i] <= d) ? 1u : 0u;
              const uint32_t pos = __reduce_add_sync(kFullMask, c);
              const uint32_t last = min(len, k - 1);  // entries [pos, last) move up by one
              for (int32_t top = (int32_t)last - 1; top >= (int32_t)pos; top -= 32) {
                const int32_t i = top - (int32_t)lane;
                float td = 0.f;
                uint32_t ti = 0;
                if (i >= (int32_t)pos) {
                  td = ld[i];
                  ti = li[i];
                }
                __syncwarp();
                if (i >= (int32_t)pos) {
                  ld[i + 1] = td;
                  li[i + 1] = ti;
                }
                __syncwarp();
              }
              if (lane == 0) {
                ld[pos] = d;
                li[pos] = id;
              }
              len = min(len + 1, k);
              __syncwarp();
            }
          }
        }
      }
      __syncthreads();
    }
    if (warp == 0) {
      for (uint32_t i = lane; i < k; i += 32) {
        const size_t o = (size_t)q * k + i;
        if (i < len) {
          out_rows[o] = ix.row_ids[li[i]];
          if (out_nodes) out_nodes[o] = li[i];
          out_dist[o] = ld[i];
        } else {
          out_rows[o] = 0xFFFFFFFFFFFFFFFFull;
          if (out_nodes) out_nodes[o] = kInvalid;
          out_dist[o] = INFINITY;
        }
      }
      if (lane == 0) out_counts[q] = len;
    }
  }
}

}  // namespace turdb
